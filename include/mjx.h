/* mjx — C ABI of the B200-native batched riichi self-play environment (libmjx.so).
 *
 * This is the drop-in boundary for libriichi's self-play hot path. libriichi has no C ABI of its
 * own (it is Rust re-exported through PyO3); each entry point below names the reference interface
 * it stands in for (paths relative to /root/reference/libriichi/src). Plain pointers and sizes only;
 * "dev" pointers are CUDA device pointers (e.g. torch.Tensor.data_ptr()), "host" pointers are
 * ordinary host memory; `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 * Every function returns 0 on success or a negative mjx_status; mjx_last_error() gives the text.
 * There is no CPU fallback: without a CUDA device every call fails with MJX_ERR_CUDA.
 */
#ifndef MJX_H
#define MJX_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum mjx_status { MJX_OK = 0, MJX_ERR_CUDA = -1, MJX_ERR_ARG = -2, MJX_ERR_TABLES = -3, MJX_ERR_STATE = -4 };

#define MJX_ACTION_SPACE 46      /* consts.rs:7-15 */
#define MJX_OBS_COLS 34
#define MJX_MAX_ROWS_PER_TABLE 3 /* <=3 seats can act on one event; a kan-select pass adds a row to 1 */

typedef struct mjx_env mjx_env;

const char* mjx_last_error(void);

/* lib.rs:139-140 (shanten::ensure_init / agari::ensure_init): load the three lookup tables from
 * `data_dir` (shanten_suhai.bin, shanten_jihai.bin, agari.bin) into device memory of `device`. */
int mjx_init(const char* data_dir, int device);

/* consts.rs:20-28 obs_shape(version).0 ; returns <0 for an unsupported version. */
int mjx_obs_rows(int version);

/* ---- environment: arena/game.rs:230-316 BatchGame::run over n_tables Game objects -------------
 * seeds: host arrays (nonce, key) per table = GameResult.seed (arena/one_vs_three.rs:140-142).
 * shuffle_kind: 0 = rand 0.9.1 (Cargo.lock:1042), 1 = rand 0.8 (the shipped seeded log).
 * enable_quick_eval: agent/mortal.rs:210-242. obs_version: consts.rs MAX_VERSION (4 supported). */
int mjx_env_create(mjx_env** out, int n_tables, const uint64_t* nonces_host, const uint64_t* keys_host,
                   int obs_version, int shuffle_kind, int enable_quick_eval);
void mjx_env_destroy(mjx_env* env);

/* One BatchGame::run loop iteration for every live table (game.rs:286-304): commit the actions
 * chosen for the rows of the previous step (agent/mortal.rs:292-573 decode + board.rs:524-533
 * validation), then poll every table to its next decision point (game.rs:59-178) and emit the
 * decision rows + legal masks (agent/mortal.rs:200-290). `actions_dev` = int64 [row_cap], indexed
 * by the previous step's row numbers (ignored on the first step; may be NULL then).
 * `q_values_dev` = float32 [row_cap, 46] Q-values of those rows, or NULL; only read for seats whose engine
 * set enable_rule_based_agari_guard (agent/mortal.rs:319-336: "wants agari but the guard objects -> best other Q"). */
int mjx_env_step(mjx_env* env, const int64_t* actions_dev, const float* q_values_dev, void* stream);

/* agent/mortal.rs:54-74, 210-250: enable_quick_eval is a property of the agent, so of the seat: host uint8 [n_tables, 4]
 * (NULL = the single flag given to mjx_env_create for every seat). */
int mjx_env_set_quick_eval(mjx_env* env, const uint8_t* flags_host);

/* agent/mortal.rs:61-66 enable_rule_based_agari_guard per table and seat: host uint8 [n_tables, 4] (NULL = off).
 * The guard itself is state/agent_helper.rs:262-368 rule_based_agari, evaluated on device. */
int mjx_env_set_agari_guard(mjx_env* env, const uint8_t* flags_host);

/* state/obs_repr.rs:776-790 encode_obs for every row of the current step:
 * obs_dev = float32 [row_cap, rows(version), 34] (only the first n_rows rows are written). */
int mjx_env_encode_obs(mjx_env* env, float* obs_dev, void* stream);

/* The same for a caller that holds HOST buffers (what agent/mortal.rs:126-152 hands to react_batch): encodes into the
 * device scratch `obs_dev` [row_cap, rows, 34] and copies rows [0, *n_rows) to `obs_host` (same layout) and `masks_host`
 * (uint8 [row_cap, 46]). The single-player block is computed in four row groups and the finished observations of one group drain
 * through the copy engine while the SMs work on the next. Blocking; host buffers should be pinned (cudaHostAlloc / torch
 * pin_memory) for the overlap to happen. */
int mjx_env_encode_obs_host(mjx_env* env, float* obs_dev, float* obs_host, uint8_t* masks_host, int* n_rows, void* stream);
/* The same in two halves, so that a caller can overlap the device work and the D2H copies of one batch with host work on
 * another (the libriichi.arena mirror steps two half-batches alternately): _begin enqueues everything and returns as soon as
 * *n_rows is known (it waits for the step kernel only); _finish blocks until the host buffers are complete. */
int mjx_env_encode_obs_host_begin(mjx_env* env, float* obs_dev, float* obs_host, uint8_t* masks_host, int* n_rows, void* stream);
int mjx_env_encode_obs_host_finish(mjx_env* env);

/* arena/board.rs:680-782 encode_oracle_obs for every row of the current step — the invisible observation an `is_oracle`
 * engine receives as react_batch's third argument (agent/mortal.rs:253-255; dataset/invisible.rs for the loader):
 * inv_dev = float32 [row_cap, mjx_oracle_obs_rows(version), 34]. consts.rs:30-38: 211 rows for version 1, else 217. */
int mjx_oracle_obs_rows(int version);
int mjx_env_encode_invisible(mjx_env* env, float* inv_dev, int version, void* stream);

/* Switch the observation version the encoder entry points produce (consts.rs:20-28; obs buffers must then hold
 * mjx_obs_rows(version) rows per observation). agent/mortal.rs:54-74: every agent has its own `version`; a PlayerState encodes
 * any version on request (obs_repr.rs:780). */
int mjx_env_set_obs_version(mjx_env* env, int version);

/* state/agent_helper.rs:509-593 single_player_tables (obs v4 rows 889-1011): on by default; `enable = 0`
 * leaves the block zero (the reference has no such switch; it exists for profiling the rest of the encoder).
 * mjx_env_sp_overflows: number of steps so far in which the state arena (2048 states per table on average)
 * overflowed and the blocks of that step were left zero — the reference has no such limit; it is 0 in every
 * test and benchmark here and is reported rather than hidden. */
int mjx_env_set_sp(mjx_env* env, int enable);
int mjx_env_sp_overflows(mjx_env* env, void* stream, int* n);

/* Size of the last step's single-player DP: out[0] = states, out[1] = edges, out[2..9] = states per level slot
 * (D3 W3 D2 W2 D1 W1 D0 W0). Instrumentation for profiles/ and bench.py; blocking. */
int mjx_env_sp_stats(mjx_env* env, void* stream, int* out10);

/* Blocking read-backs (synchronise `stream` first). */
int mjx_env_num_rows(mjx_env* env, void* stream, int* n_rows);          /* rows emitted by the last step */
int mjx_env_num_live(mjx_env* env, void* stream, int* n_live);          /* tables still playing */
int mjx_env_total_steps(mjx_env* env, void* stream, int64_t* steps);    /* game.rs:304 `actions` counter */

/* One blocking read-back per BatchGame::run cycle: out4 = { rows emitted by the last step, tables still playing,
 * tables that have failed so far (err != 0; game.rs:288,292 aborts the batch at that cycle, so should the caller),
 * single-player arena overflows so far (see mjx_env_sp_overflows) }. */
int mjx_env_poll(mjx_env* env, void* stream, int* out4);

/* arena/result.rs:19-51 GameResult.game_log: record every table's mjai events on device (compact 64-bit words, layout in
 * csrc/mjx_step.cuh `log_word`; mortal_b200/mjai_log.py turns them into the reference's JSON lines). Call
 * mjx_env_enable_log before the first step; `words_per_table` bounds one hanchan (a kyoku is ~170 words; 8192 is ample).
 * mjx_env_read_log copies [n_tables, words_per_table] words and the per-table counts to host (count > capacity = overflow). */
int mjx_env_enable_log(mjx_env* env, int words_per_table);
int mjx_env_read_log(mjx_env* env, void* stream, uint64_t* words_host, int32_t* len_host);
int32_t* mjx_env_log_len_dev(mjx_env* env); /* int32 [n_tables] device view of the per-table word counts (null before enable_log):
                                              read after every step it tells which events that step wrote (per-decision meta) */

/* dataset/grp.rs:90-164 without the logs: the GRP feature row of every kyoku — {grand_kyoku (E1 = 0 .. S4 = 7, W = 8+), honba,
 * kyotaku, scores[4]} as int32 (the reference's f64 row is these with the scores divided by 10000) — is written by the step
 * kernel when the kyoku starts. mjx_env_read_grp copies [n_tables, max_kyoku, 7] rows and the per-table kyoku counts (a count
 * above max_kyoku = overflow); with mjx_env_results (final scores, rank_by_player) that is everything
 * mortal/reward_calculator.py:13-38 consumes. Call mjx_env_enable_grp before the first step. */
int mjx_env_enable_grp(mjx_env* env, int max_kyoku);
int mjx_env_read_grp(mjx_env* env, void* stream, int32_t* feat_host, int32_t* n_kyoku_host);

/* ---- log replay: dataset/gameplay.rs:247-449 GameplayLoader (SURVEY.md §8f N3) ------------------------------------------
 * A job = one (game log, player). `hdr`: the games' events as 64-bit words (csrc/mjx_step.cuh `log_word`; start_game = 15,
 * end_game = 16), concatenated, job j owning ev_cnt[j] words from ev_off[j]; `kyoku`: 19 words per start_kyoku (2 of scores, 17 = the
 * 136-byte wall in board.rs:109-122 layout: the 52 dealt tiles, the rest `?` = 37 unless the hidden tiles are known),
 * job j's first payload at index ky_off[j]; `players`: the job's point of view. All host arrays. Full-information logs only.
 * mjx_env_replay_step advances every job to the next decision the log shows its player making and emits the row(s)
 * (decision, then kan-select); observation / mask / row_table / row_seat are read exactly as after mjx_env_step, plus the
 * label and (at_kyoku, at_turn, shanten, apply_gamma) of each row. A job is finished when mjx_env_num_live stops counting it. */
int mjx_env_create_replay(mjx_env** out, int n_jobs, const uint64_t* hdr, const int32_t* ev_off, const int32_t* ev_cnt, long long n_hdr,
                          const uint64_t* kyoku, const int32_t* ky_off, long long n_kyoku_words, const uint8_t* players,
                          int obs_version, int always_include_kan_select);
int mjx_env_replay_step(mjx_env* env, void* stream);
/* dataset/invisible.rs:35-66 (`trust_seed`): the logs were produced from known seeds (start_game.seed, what this arena and
 * libriichi's write) — host arrays (nonce, key) per job. Every kyoku's wall is then regenerated on device (board.rs:99-123), checked
 * against the logged haipai / dora marker (a mismatch fails the job), and mjx_env_encode_invisible can show the hidden tiles.
 * Call before the first mjx_env_replay_step. */
int mjx_env_replay_trust_seeds(mjx_env* env, const uint64_t* nonces_host, const uint64_t* keys_host, int shuffle_kind);
int64_t* mjx_env_row_label(mjx_env* env); /* int64 [row_cap] device */
uint8_t* mjx_env_row_meta(mjx_env* env);  /* uint8 [row_cap, 4] device: at_kyoku, at_turn, shanten (int8), apply_gamma */

/* ---- libriichi.state.PlayerState (state/player_state.rs:143-264, state/getter.rs:6-156, state/obs_repr.rs:776-791) ---------
 * A batch of n independent single-seat states: table records in single-seat mode (other seats' hidden tiles are `?` = 37), updated
 * by the same device event handlers self-play uses. `mjx_state_create` returns an mjx_env whose encoder entry points
 * (mjx_env_encode_obs, mjx_env_masks, mjx_env_encode_obs_host ...) work on the rows mjx_state_rows prepares.
 *   mjx_state_update  PlayerState::update (update.rs:24-122): one event per state as a 64-bit word (csrc/mjx_step.cuh log_word;
 *                     mortal_b200/dataset_codec.py encodes mjai JSON), start_kyoku with its 19-word payload (scores + wall, see
 *                     mjx_env_create_replay); word 0 = no event for that state. cans_host[i] = the ActionCandidate of state i
 *                     (action.rs:11-40: bit k = the k-th can_* flag in declaration order, target_actor << 16).
 *   mjx_state_view    every getter of state/getter.rs plus the fields state/test.rs asserts, for one state.
 *   mjx_state_rows    one decision row per state (kan-select rows where at_kan_select_host[i] != 0): row i = state i.
 *   mjx_state_query   what = 0 agent_helper.rs:377-462 agari_points(is_ron = args[0], ura tiles args[2 .. 2 + args[1]))
 *                              -> out = {ron, tsumo_ko, tsumo_oya, ok};  1 rule_based_agari (agent_helper.rs:262-368) -> out[0];
 *                     2 discard_candidates_aka (agent_helper.rs:35-79) -> out[0..1] = 37-bit mask (low, high word);
 *                     3 discard_candidates_with_unconditional_tenpai (agent_helper.rs:88-197) -> 34-bit mask;
 *                     4 agent/mortal.rs:338-573 action id -> reaction: args = {action, kan_select_action or -1}
 *                              -> out[0..1] = the event word (low, high), out[2] = 0 or an error code. */
typedef struct mjx_player_view {
    uint8_t tehai[34], waits[34], dora_factor[34], tiles_seen[34], keep_shanten_discards[34], next_shanten_discards[34],
        forbidden_tiles[34], discarded_tiles[34];
    uint8_t akas_seen[3], akas_in_hand[3];
    uint8_t bakaze, jikaze, kyoku, honba, kyotaku, rank, oya, is_all_last;
    int32_t scores[4];                       /* rotated: [0] = self */
    uint8_t n_dora_indicators, dora_indicators[5];
    uint8_t riichi_declared[4], riichi_accepted[4];  /* relative seats */
    uint8_t at_turn, tiles_left;
    int8_t shanten, real_time_shanten;
    uint8_t has_last_self_tsumo, last_self_tsumo, has_last_kawa_tile, last_kawa_tile;
    uint32_t cans;
    uint8_t n_ankan_candidates, ankan_candidates[3], n_kakan_candidates, kakan_candidates[3];
    uint8_t chankan_chance, can_w_riichi, is_w_riichi, at_rinshan, at_ippatsu, at_furiten, to_mark_same_cycle_furiten,
        kans_on_board, is_menzen;
    uint8_t n_chis, chis[4], n_pons, pons[4], n_minkans, minkans[4], n_ankans, ankans[4];
    uint8_t doras_owned[4], doras_seen, tehai_len_div3, has_next_shanten_discard;
    uint8_t kawa_len[4];
    uint8_t viewer, pad_[3];
    int32_t err;                             /* 0, or the code of the inconsistency the last events produced */
} mjx_player_view;
int mjx_state_create(mjx_env** out, int n, const uint8_t* player_ids_host, int obs_version);
int mjx_state_update(mjx_env* env, const uint64_t* words_host, const uint64_t* payload_host, uint32_t* cans_host);
int mjx_state_view(mjx_env* env, int index, mjx_player_view* out_host);
int mjx_state_rows(mjx_env* env, const uint8_t* at_kan_select_host, void* stream);
int mjx_state_query(mjx_env* env, int index, int what, const int32_t* args, int32_t* out);
int mjx_state_copy(mjx_env* dst, int dst_index, mjx_env* src, int src_index); /* PlayerState: Clone */

/* Instrumentation for bench.py's roofline: when enabled, mjx_env_encode_obs brackets its two encoder kernels with CUDA events
 * on the launch stream; mjx_env_last_encode_ms (blocking) returns the durations of k_encode_features and k_encode_store. */
int mjx_env_set_encode_timing(mjx_env* env, int enable);
int mjx_env_last_encode_ms(mjx_env* env, float* ms_features, float* ms_store);

/* Number of kernels this library has launched for env so far (host-side counter; bench.py's gpu_launches). */
long long mjx_env_launch_count(mjx_env* env);

/* Device views, valid for the lifetime of env (contents valid until the next mjx_env_step). */
int mjx_env_row_cap(mjx_env* env);
uint8_t* mjx_env_masks(mjx_env* env);      /* uint8/bool [row_cap, 46]  (obs_repr.rs mask) */
int32_t* mjx_env_row_table(mjx_env* env);  /* int32 [row_cap] table index of each row */
uint8_t* mjx_env_row_seat(mjx_env* env);   /* uint8 [row_cap] seat | (kan_select << 2) */
uint32_t* mjx_env_row_step(mjx_env* env); /* uint32 [row_cap] table-step index of the table when the row was emitted */
int32_t* mjx_env_num_rows_dev(mjx_env* env); /* int32 [1] */

/* arena/result.rs GameResult.scores + rankings.rs rank_by_player, plus per-table step counts and
 * error codes (0 = clean; the reference would have raised/panicked otherwise). Host outputs. */
int mjx_env_results(mjx_env* env, void* stream, int32_t* scores_host /*[n,4]*/, uint8_t* ranks_host /*[n,4]*/,
                    int32_t* steps_host /*[n]*/, int32_t* err_host /*[n]*/, int32_t* done_host /*[n]*/);

/* Counter-based TEST policy (not in the reference; shared definition with the oracle) writing
 * int64 actions for the current rows. kind 0 uniform, 1 agari-first/shanten-greedy.
 * trace_dev (optional): int64 [row_cap, 6] = table, step, seat, action, kan_select, mask_bits.
 * q_values_dev (optional): float32 [row_cap, 46] filled with 0 on legal and -inf on illegal actions. */
int mjx_env_policy_test(mjx_env* env, int kind, int64_t* actions_dev, int64_t* trace_dev, float* q_values_dev,
                        void* stream);

/* ---- policy-net inference helpers (not part of libriichi's surface; mortal/model.py ResBlock + ChannelAttention) ------------
 * Fused elementwise passes between the cuDNN convolutions: bf16 channels-last activations [batch, length, channels]
 * (device pointers, 16-byte aligned, channels % 8 == 0), fp32 math. scale/bias = eval-mode BatchNorm folded to an affine. */
int mjx_nn_affine_mish_bf16(const void* x, const float* scale, const float* bias, void* out, long long n_elems, int channels,
                            void* stream);                                   /* out = mish(x * scale[c] + bias[c]) */
int mjx_nn_pool_bf16(const void* x, void* avg, void* mx, int batch, int length, int channels, void* stream);  /* [batch, channels] each */
int mjx_nn_gate_residual_bf16(const void* y, const void* gate, const void* x, void* out, int batch, int length, int channels,
                              void* stream);                                 /* out = y * gate[b, c] + x */
/* observations f32 [batch, channels, length] -> bf16 channels-last [batch, length, channels_padded], padded channels zero
 * (channels_padded % 64 == 0): the input of the stem convolution. */
int mjx_nn_obs_to_nhwc_bf16(const float* obs, void* out, int batch, int channels, int length, int channels_padded, void* stream);
/* The tail of a residual block and the next pre-activation in one pass (model.py ChannelAttention + residual; next BN + Mish):
 * gate = sigmoid(mlp(mean_l y) + mlp(max_l y)), mlp = w2 . mish(w1 [hidden, channels] . v + b1) + b2, w2 passed TRANSPOSED as w2t
 * [hidden, channels] (fp32 device
 * arrays); x_out = y * gate + x; a_out = mish(x_out * scale[c] + bias[c]). Two launches: one warp per batch row computes the gate,
 * one streaming pass applies it. channels % 8 == 0, <= 256. */
int mjx_nn_block_tail_bf16(const void* y, const void* x, const float* w1, const float* b1, const float* w2t, const float* b2,
                           const float* scale, const float* bias, void* gate_scratch /* bf16 [batch, channels] */, void* x_out,
                           void* a_out, int batch, int length, int channels, int hidden, void* stream);

/* mjx_nn_obs_to_nhwc_bf16 of a gathered batch: output row i is observation rows[i] for i < *count_dev, zeros for the rest of
 * `batch` (rows, count_dev: device int32). */
int mjx_nn_obs_rows_to_nhwc_bf16(const float* obs, const int* rows, const int* count_dev, void* out, int batch, int channels, int length,
                                 int channels_padded, void* stream);

/* ---- action selection on the device path (mortal/engine.py MortalEngine._react_batch + mortal/model.py DQN.forward) --------------
 * Batch row i < min(*count_dev, n_max) is environment row r = rows[i] (rows NULL: r = i); v f32 [n] and a f32 [n, 46] with row strides.
 * Writes q_out[r] (dueling Q, -inf on illegal actions per masks[r]), actions[r] (int64) and greedy[r] (uint8, optional): the argmax
 * (lowest index on ties), or with probability epsilon a draw from softmax(q / temp) over the top-p nucleus of the legal actions.
 * Randomness: Philox4x32-10 with key `seed` and counter (table_offset + row_table[r], row_step[r], row_seat[r]), so a decision's
 * draw does not depend on the order of the rows. */
int mjx_select_actions(const float* v, long long v_stride, const float* a, long long a_stride, const int* rows, const int* count_dev,
                       int n_max, const void* masks, const int* row_table, const uint32_t* row_step, const uint8_t* row_seat,
                       unsigned long long seed, int table_offset, float epsilon, float temp, float top_p, int64_t* actions,
                       float* q_out, uint8_t* greedy, void* stream);
/* Stable split of the step's *count_dev rows by agent_of[row_table * 4 + (row_seat & 3)] (0 or 1): rows0 / rows1 get the row indices
 * in order, counts[0..1] (device int32) their numbers. One CTA. */
int mjx_split_rows(const int* row_table, const uint8_t* row_seat, const int* count_dev, const uint8_t* agent_of, int* rows0, int* rows1,
                   int* counts, void* stream);

/* ---- standalone kernels (BASELINE configs 3/4) ------------------------------------------------ */
/* algo/shanten.rs:138-150 calc_all: tiles_dev uint8 [n,34], len_div3_dev uint8 [n] -> int8 [n]. */
int mjx_shanten(const uint8_t* tiles_dev, const uint8_t* len_div3_dev, int8_t* out_dev, int n, void* stream);

typedef struct mjx_agari_in {  /* algo/agari.rs:77-101 AgariCalculator */
    uint8_t tehai[34];
    uint8_t chis[4], pons[4], minkans[4], ankans[4];
    uint8_t n_chis, n_pons, n_minkans, n_ankans;
    uint8_t bakaze, jikaze, winning_tile, is_ron;
    uint8_t additional_hans, doras; /* for mode 1 = agari(additional_hans, doras) */
    uint8_t is_oya, pad;
} mjx_agari_in;
typedef struct mjx_agari_out { /* algo/agari.rs:66-74 Agari + algo/point.rs Point */
    uint8_t kind; /* 0 none, 1 normal, 2 yakuman */
    uint8_t fu, han, yakuman;
    int32_t ron, tsumo_ko, tsumo_oya; /* -1 where point.rs would panic */
} mjx_agari_out;
/* mode 0 = search_yakus (agari.rs:212), 1 = agari (agari.rs:225), 2 = has_yaku (agari.rs:206),
 * 3 = check_ankan_after_riichi(tehai, len_div3 = additional_hans, tile = winning_tile, strict = false) (agari.rs:854-912;
 *     the call state/update.rs:278 makes): out.kind = 1 when the kan is allowed */
int mjx_agari(const mjx_agari_in* in_dev, mjx_agari_out* out_dev, int n, int mode, void* stream);

/* Host-buffer conveniences (H2D + kernel + D2H), the shape a foreign-language binding would call. */
int mjx_shanten_host(const uint8_t* tiles, const uint8_t* len_div3, int8_t* out, int n);
int mjx_agari_host(const mjx_agari_in* in, mjx_agari_out* out, int n, int mode);

/* arena/board.rs:99-123 wall for one (seed, kyoku, honba): uint8 [136] (host out; runs on device). */
int mjx_make_wall_host(uint64_t nonce, uint64_t key, int kyoku, int honba, int shuffle_kind, uint8_t* wall136);

#ifdef __cplusplus
}
#endif
#endif /* MJX_H */
