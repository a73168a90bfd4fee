/* toybox_b200.h -- C ABI of libtoybox_b200.so: a batched, device-resident replacement for the part of
 * `ctoybox` (pinned ==0.5.0, /root/reference/REQUIREMENTS.txt:12) that the reference drives on its hot
 * path.  One `tbx_pool` holds N independent environments of one game on one CUDA device; every call
 * below is the batched restatement of a ctoybox entry point.  The reference reaches those entry
 * points through the `ctoybox.Toybox` python shim; the call sites that each function replaces are
 * cited per declaration (paths relative to /root/reference).
 *
 * Conventions
 *   - every function returns 0 on success and a non-zero TBX_E* code on failure; it never throws or
 *     aborts across the ABI.  tbx_last_error() returns a thread-local description of the last failure.
 *   - pointers named *_dev are CUDA device pointers on the pool's device (e.g. torch.Tensor.data_ptr());
 *     pointers named *_host are ordinary host memory.  Buffers are caller-owned unless stated otherwise.
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream).  Device work is
 *     enqueued on it and NOT synchronised unless stated otherwise.
 *   - a pool is used by one host thread at a time (same rule as a ctoybox handle).
 */
#ifndef TOYBOX_B200_H
#define TOYBOX_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tbx_pool tbx_pool;

enum { TBX_OK = 0, TBX_EINVAL = 1, TBX_ECUDA = 2, TBX_EJSON = 3, TBX_ENOMEM = 4, TBX_EACTION = 5 };

/* observation layouts written by tbx_render (H, W = the game's native frame size) */
enum {
  TBX_OBS_RGBA = 0,  /* uint8[N][H][W][4]  Toybox.get_state() with grayscale=False  (envs/atari/base.py:109) */
  TBX_OBS_RGB = 1,   /* uint8[N][H][W][3]  Toybox.get_rgb_frame()                   (envs/atari/base.py:164) */
  TBX_OBS_GRAY = 2,  /* uint8[N][H][W]     Toybox.get_state() with grayscale=True   (envs/atari/base.py:109) */
  TBX_OBS_GRAY_AREA = 3, /* uint8[N][out_h][out_w]  cv2.resize(gray, (out_w,out_h), INTER_AREA) = baselines WarpFrame
                           (baselines/baselines/common/atari_wrappers.py:230-244), fused into the render */
  TBX_OBS_RGB_AREA = 4  /* uint8[N][out_h][out_w][3]  cv2.resize(get_rgb_frame(), (out_w,out_h), INTER_AREA): WarpFrame(grayscale=False),
                           64x64 / 84x84 colour observations; the same output sizes as TBX_OBS_GRAY_AREA */
};

const char *tbx_last_error(void);
int tbx_version(void);

/* ---- simulator_alloc(name) + state_alloc: Toybox(game_name) ctor (envs/atari/breakout.py:6-11 etc.).
 * game: "breakout" | "amidar" | "space_invaders".  cfg_json: NULL for the default config, else a config
 * in the schema of Toybox.config_to_json().  All envs start from the default simulator rand and
 * new_game(), i.e. each is exactly the state a fresh ctoybox.Toybox(game) holds. */
int tbx_pool_create(const char *game, int n_envs, int device, const char *cfg_json, tbx_pool **out);
/* simulator_free + state_free */
int tbx_pool_destroy(tbx_pool *pool);

/* simulator_frame_width / simulator_frame_height: Toybox.get_width()/get_height() (envs/atari/base.py:64-66) */
int tbx_frame_width(const tbx_pool *pool);
int tbx_frame_height(const tbx_pool *pool);
int tbx_n_envs(const tbx_pool *pool);
int tbx_device(const tbx_pool *pool);
/* simulator_actions: Toybox.get_legal_action_set() (envs/atari/base.py:57).  Writes up to cap ids, returns the count. */
int tbx_legal_actions(const tbx_pool *pool, int32_t *out_host, int cap);
/* bytes of one env's observation in the given layout (0 if the layout/size is unsupported) */
size_t tbx_obs_bytes(const tbx_pool *pool, int obs_mode, int out_w, int out_h);

/* simulator_seed: Toybox.set_seed(seed) (envs/atari/base.py:95).  Sets the simulator-level rand of the
 * listed envs (env_ids_host == NULL: envs 0..n-1 get seeds_host[0..n-1]).  Like ctoybox it does not
 * start a new game.  Synchronous. */
int tbx_seed(tbx_pool *pool, const uint32_t *seeds_host, const int32_t *env_ids_host, int n);

/* Toybox.new_game() (envs/atari/base.py:97,153; interventions/base.py:403).  mask_dev == NULL: every env;
 * else uint8[N], non-zero = reset that env. */
int tbx_new_game(tbx_pool *pool, const uint8_t *mask_dev, void *stream);

/* state_apply_ale_action: Toybox.apply_ale_action(id) for every env (envs/atari/base.py:126), fused with the
 * env-level bookkeeping of ToyboxBaseEnv.step (base.py:136-147): reward = max(score - prev_score, 0),
 * done = lives <= 0, and, if auto_reset != 0, new_game() for finished envs as the reference's vectorised
 * driver does (baselines/baselines/common/vec_env/subproc_vec_env.py:11-15).
 * actions_dev: int32[N] ALE action ids.  Outputs (each may be NULL): reward int32[N], done uint8[N],
 * score int32[N], lives int32[N] -- score/lives are the values BEFORE an auto-reset.
 * An id outside 0..17 leaves that env untouched and is reported by the next tbx_check(). */
int tbx_step(tbx_pool *pool, const int32_t *actions_dev, int auto_reset, int32_t *reward_dev, uint8_t *done_dev,
             int32_t *score_dev, int32_t *lives_dev, void *stream);
/* state_apply_action: Toybox.apply_action(Input) (test/interventions/test_breakout_interventions.py:12-15).
 * inputs_dev: uint8[N] bitmask left=1 right=2 up=4 down=8 button1=16 button2=32. */
int tbx_step_inputs(tbx_pool *pool, const uint8_t *inputs_dev, int auto_reset, int32_t *reward_dev, uint8_t *done_dev,
                    int32_t *score_dev, int32_t *lives_dev, void *stream);
/* The same step driven by the benchmark's synthetic action stream (tbx_fill_actions below), generated inside the step kernel:
 * env i takes legal[index(seed, env0 + i, t)].  One launch instead of two; bit-identical to tbx_fill_actions + tbx_step. */
int tbx_step_random(tbx_pool *pool, uint64_t seed, uint64_t env0, uint64_t t, int auto_reset, int32_t *reward_dev, uint8_t *done_dev,
                    int32_t *score_dev, int32_t *lives_dev, void *stream);
/* synchronises `stream` and returns TBX_EACTION if any env received an invalid action id since the last check, else
 * TBX_EINVAL if a state snapshot load or save skipped entries (tbx_state_load below) since the last check */
int tbx_check(tbx_pool *pool, void *stream);

/* render_current_frame: Toybox.get_state() / get_rgb_frame() for every env (envs/atari/base.py:109,164).
 * dst_dev: N * tbx_obs_bytes() bytes, 16-byte aligned.  out_w/out_h are used by TBX_OBS_GRAY_AREA and TBX_OBS_RGB_AREA only. */
int tbx_render(tbx_pool *pool, uint8_t *dst_dev, int obs_mode, int out_w, int out_h, void *stream);

/* state_lives / state_score / state_level / state_game_over (envs/atari/base.py:20-27,136,145).  Device
 * outputs, each may be NULL. */
int tbx_read_scalars(tbx_pool *pool, int32_t *score_dev, int32_t *lives_dev, int32_t *level_dev, void *stream);

/* One whole env.step() for callers that live on the host (the reference's own calling convention):
 * copies actions_host (int32[N]) to the device, steps, renders, and copies observations and scalars back
 * into host buffers (pinned memory makes the copies asynchronous to each other); returns when they have
 * landed.  Any output pointer may be NULL. */
int tbx_step_host(tbx_pool *pool, const int32_t *actions_host, int auto_reset, int obs_mode, int out_w, int out_h,
                  uint8_t *obs_host, int32_t *reward_host, uint8_t *done_host, int32_t *score_host, int32_t *lives_host);

/* state_to_json / state_from_json: Toybox.to_state_json() / write_state_json() (interventions/base.py:391,406)
 * for the listed envs.  out_json[k] is malloc'ed by the library; release with tbx_free_str.  Synchronous. */
int tbx_state_to_json(tbx_pool *pool, const int32_t *env_ids_host, int n, char **out_json);
int tbx_state_from_json(tbx_pool *pool, const int32_t *env_ids_host, int n, const char *const *json);
/* simulator_to_json / simulator_from_json: Toybox.config_to_json() / write_config_json() (interventions/base.py:390,402).
 * As in ctoybox a new config takes effect at the next new_game(). */
int tbx_config_to_json(tbx_pool *pool, char **out_json);
int tbx_config_from_json(tbx_pool *pool, const char *json);
/* simulator_schema_for_state / simulator_schema_for_config: Toybox.schema_for_state() (interventions/breakout.py:38-41) */
int tbx_schema_for_state(const char *game, char **out_json);
int tbx_schema_for_config(const char *game, char **out_json);
/* state_query_json: Toybox.query_state_json(query, args) (interventions/amidar.py:508-518) for one env */
int tbx_query_json(tbx_pool *pool, int env_id, const char *query, const char *args_json, char **out_json);
void tbx_free_str(char *s);

/* BreakoutIntervention.add_channel(col) / fill_column(col) (toybox/interventions/breakout.py:406-416) and the channel count
 * behind rstate.breakout_channel_count() (baselines/baselines/run_get_seed_state.py:266-270) for every env in one launch:
 * op 0 = the bricks of column `col` dead, 1 = alive again (mask_dev, uint8[N] or NULL, selects the envs), 2 = out_dev[env] =
 * columns with no alive brick (int32[N]).  Columns follow each env's own brick table (bricks[i].col). */
int tbx_breakout_columns(tbx_pool *pool, int op, int col, const uint8_t *mask_dev, int32_t *out_dev, void *stream);

/* Episode statistics accumulated on the device since the last reset of the counters (the role of
 * baselines/baselines/bench/monitor.py:58-76): out_host[0..3] = episodes finished, sum of episode returns,
 * sum of episode lengths, max episode return.  This 32-byte vector is what the multi-GPU driver all-reduces. */
int tbx_stats_read(tbx_pool *pool, int64_t *out_host, int reset, void *stream);
/* The same vector copied device-to-device into out_dev (int64[4]) in stream order, no host synchronisation: the form the
 * NCCL all-reduce of a multi-GPU rollout consumes (toybox_b200/distributed.py, bench.py). */
int tbx_stats_read_device(tbx_pool *pool, int64_t *out_dev, void *stream);

/* The synthetic random-action stream of the benchmark and parity tests: fills actions_dev[i] with
 * legal[index(seed, env0 + i, t)] for the pool's game (counter-based, reproducible on the CPU). */
int tbx_fill_actions(tbx_pool *pool, int32_t *actions_dev, uint64_t seed, uint64_t env0, uint64_t t, void *stream);
/* The same with the frame counter t read from device memory (*t_dev) when the kernel runs: a CUDA graph that captured
 * fill + step + render then advances the action stream on every replay (the caller increments *t_dev in the graph). */
int tbx_fill_actions_at(tbx_pool *pool, int32_t *actions_dev, uint64_t seed, uint64_t env0, const uint64_t *t_dev, void *stream);

/* Benchmark utility: scripted actions computed on the device from the envs' own state.  policy 1 = Breakout
 * "track the ball" (FIRE to serve, then follow the first ball with a varying aim offset), which drives games deep
 * into the brick wall -- states the uniform random stream almost never reaches. */
int tbx_fill_actions_policy(tbx_pool *pool, int32_t *actions_dev, int policy, uint64_t t, void *stream);

/* ---- Vectorised property access (SURVEY 8 f3): one scalar of the JSON state schema for EVERY env without a JSON round
 * trip.  Replaces, at batch size N, get_property / set-through-Intervention on one env
 * (toybox/interventions/core.py:271-304, base.py:387-408) and the per-game helpers built on them
 * (interventions/breakout.py:303-429, amidar.py:406-481).  `path` uses the schema's names: "lives", "score",
 * "paddle.position.x", "balls[0].velocity.y", "bricks[17].alive", "ufo.appearance_counter", "enemies[3].alive",
 * "player.position.x", "jump_timer", "board.boxes[4].painted", ...  kind: 0 int32, 1 float64, 2 bool, 3 bool stored as
 * one bit, 4 Option<i32> (null <-> INT32_MIN).  Values travel as int32[N] (kinds 0, 2, 3, 4) or float64[N] (kind 1)
 * device arrays; mask_dev (may be NULL) = uint8[N], only flagged envs are written.  Setting "score" also sets the
 * env's reward baseline, as tbx_state_from_json does. */
int tbx_field_lookup(const char *game, const char *path, int *word, int *kind, int *bit);
int tbx_field_get(tbx_pool *pool, const char *path, void *out_dev, void *stream);
int tbx_field_set(tbx_pool *pool, const char *path, const void *values_dev, const uint8_t *mask_dev, void *stream);

/* ---- The DeepMind-style wrapper stack of the reference's trainers, fused (SURVEY 8(f1)).
 * Replaces, per agent step and for every env at once, the Python chain
 *   make_atari:    MaxAndSkipEnv(NoopResetEnv(env, noop_max=30), skip=4)     baselines/baselines/common/atari_wrappers.py:107-134,186-209,323-333
 *   wrap_deepmind: FrameStack(ClipRewardEnv(WarpFrame(FireResetEnv(EpisodicLifeEnv(env)))), 4)   :136-184,211-244,246-275,345-360
 * plus the reset-on-done of the VecEnv worker (vec_env/subproc_vec_env.py:11-15).  One kernel runs the `skip`
 * transitions of an agent step (and the whole reset sequence of finished envs); one render pass draws the two states
 * whose pixel-wise max, down-sampled with INTER_AREA to out_w x out_h, is the observation.
 * Each of episodic_life / fire_reset / clip_rewards is 0 or 1 (the wrap_deepmind switches); noop_max 0 = no
 * NoopResetEnv.  The no-op count of reset r of env i is 1 + tbx action-stream index(noop_seed, env0 + i, r, noop_max). */
typedef struct tbx_wrap tbx_wrap;
int tbx_wrap_create(tbx_pool *pool, int skip, int noop_max, int episodic_life, int fire_reset, int clip_rewards, int stack_k,
                    int out_w, int out_h, uint64_t noop_seed, uint64_t env0, tbx_wrap **out);
/* What a reset observation does to the other k-1 slots of an env's ring: 0 (default) = it fills them, FrameStack.reset
 * (baselines/baselines/common/atari_wrappers.py:262-266, the wrap_deepmind(frame_stack=True) path); 1 = they are zeroed,
 * VecFrameStack (baselines/baselines/common/vec_env/vec_frame_stack.py:17-30, the make_vec_env + VecFrameStack path). */
int tbx_wrap_set_stack_mode(tbx_wrap *w, int mode);
/* The layout of the observation ring: TBX_OBS_GRAY_AREA (default; the ring is uint8[N][stack_k][out_h][out_w]) or
 * TBX_OBS_RGB_AREA, WarpFrame(grayscale=False) (atari_wrappers.py:230-244): the ring is uint8[N][stack_k][out_h][out_w][3],
 * each observation the colour INTER_AREA down-sample of the pixel-wise max of the two RGB frames.  Both accept the same
 * output sizes.  TBX_EINVAL for any other layout, or once the wrap has stepped (its ring holds frames of the old layout). */
int tbx_wrap_set_obs_mode(tbx_wrap *w, int obs_mode);
/* Device buffers (int32[N] each, caller-owned, may be NULL) that every tbx_wrap_step fills with baselines' Monitor record
 * (bench/monitor.py:58-76; Monitor sits between make_atari and wrap_deepmind, common/cmd_util.py:30-36) of the episode that
 * ended in that agent step: r = sum of raw rewards, l = MaxAndSkipEnv steps since the last real reset.  Valid where real_done
 * or truncated (tbx_wrap_set_time_limit). */
int tbx_wrap_set_episode_outputs(tbx_wrap *w, int32_t *ep_return_dev, int32_t *ep_length_dev);
/* Sticky actions (repeat_action_probability p, ALE's `if (rand() >= p) m_player_a_action = action`): on every game frame the
 * stack runs -- the skipped frames, the no-ops of NoopResetEnv, the FIRE / RIGHT steps of FireResetEnv, the NOOP step of a
 * life-loss reset -- env i repeats the ALE id of its previous frame where the draw u of (seed, env0 + i, f) is below
 * llround(p * 2^32), else applies the requested id.  u is the upper 32 bits of the splitmix64 mix of the action stream, keyed
 * with seed ^ 0x5354494B59414354; f counts env i's frames and is never reset; a new game sets the remembered id to NOOP.
 * p > 0 adds two wrapper words per env (remembered id, frame counter: tbx_wrap_state_rows grows by 2), p = 0 (default) turns
 * the rule off.  TBX_EINVAL for p outside [0, 1] or NaN, or once the wrap has stepped. */
int tbx_wrap_set_sticky_actions(tbx_wrap *w, double repeat_action_probability, uint64_t seed);
/* Episode time limit (gym's TimeLimit between MaxAndSkipEnv and Monitor): an env whose Monitor length (MaxAndSkipEnv steps since
 * the last real reset, reset-chain steps included) reaches max_episode_steps at the end of an agent step reports done, takes
 * the full reset chain and exports its Monitor record; truncated_dev (uint8[N], caller-owned, may be NULL; written on every
 * step) flags such an env where its game is not over.  real_done keeps meaning game over.  Reset-chain steps that cross the
 * limit truncate at the next agent step.  0 (default) = no limit.  TBX_EINVAL for a negative limit, or once the wrap has
 * stepped. */
int tbx_wrap_set_time_limit(tbx_wrap *w, int max_episode_steps, uint8_t *truncated_dev);
int tbx_wrap_destroy(tbx_wrap *wrap);
/* env.step(action) of the wrapped env for every env (actions_dev: int32[N] gym action indices into the legal set), or
 * env.reset() for every env when actions_dev == NULL.  obs_ring_dev: uint8[N][stack_k][out_h][out_w] (with [3] appended
 * under TBX_OBS_RGB_AREA, tbx_wrap_set_obs_mode), a ring of the
 * last stack_k observations per env; the newest frame goes to slot *slot_out (host int), older frames follow
 * backwards modulo stack_k (FrameStack order = slots slot+1, ..., slot+stack_k, modulo stack_k).  Envs whose
 * observation comes from a reset get it in every slot (FrameStack.reset).  reward: sum over the skipped frames,
 * its sign when clip_rewards; done: as the agent sees it (game over, a lost life when episodic_life, or the time limit);
 * real_done: game over; score / lives: before any reset.  Output pointers may be NULL. */
int tbx_wrap_step(tbx_wrap *wrap, const int32_t *actions_dev, uint8_t *obs_ring_dev, int32_t *reward_dev, uint8_t *done_dev,
                  uint8_t *real_done_dev, int32_t *score_dev, int32_t *lives_dev, int *slot_out, void *stream);

/* ---- Device-resident state snapshots: save, restore and fork envs without the JSON codec (DESIGN.md 4.7).
 * A snapshot of k envs is a caller-owned device buffer uint32[rows][k], word-major like the pool's planes: column j is one
 * env's whole record (both rngs, prev_score, the episode counters; rows = tbx_state_rows), followed for a wrapped env by its
 * 5 wrapper words (EpisodicLife lives, was_real_done, reset counter, Monitor return, Monitor length), 7 with sticky actions
 * (+ the remembered ALE id and the frame counter); rows = tbx_wrap_state_rows.  A loaded env continues exactly as the saved env would have.  The device-wide episode statistics
 * (tbx_stats_read) are pool state and are neither saved nor restored.
 * Breakout and Amidar records index the pool's geometry tables, so a snapshot goes with the tables blob of the moment it was
 * saved (tbx_state_tables): a tbx_state_blob_header followed by table_count tables of table_bytes bytes each (none for Space
 * Invaders).  Tables are only ever appended, so every index in a snapshot is below the count exported after saving it.
 * Snapshots are trusted binary data written by tbx_state_save: a load checks the blob's header on the host (a mismatch returns
 * TBX_EINVAL before any device work and leaves the pool unchanged) and, on the device, each entry's env id, column and table
 * index; an entry out of range is skipped and counted, and the next tbx_check returns TBX_EINVAL with the count.  No other field
 * is re-validated -- to_state_json / write_state_json stay the validated import. */
#define TBX_STATE_MAGIC 0x53584254u /* "TBXS" */
#define TBX_STATE_FORMAT 1          /* the record layout; a snapshot of another format is refused */
typedef struct {
  uint32_t magic, format;
  uint32_t game;        /* 0 breakout, 1 amidar, 2 space_invaders */
  uint32_t rows;        /* rows of the snapshot this blob belongs to */
  uint32_t table_bytes; /* bytes of one geometry table */
  uint32_t table_count;
} tbx_state_blob_header;
int tbx_state_rows(const tbx_pool *pool);
int tbx_wrap_state_rows(const tbx_wrap *wrap);
/* *size = bytes of the blob; it is written to out_host when out_host != NULL (TBX_EINVAL if cap < *size).  Host only. */
int tbx_state_tables(const tbx_pool *pool, void *out_host, size_t cap, size_t *size);
int tbx_wrap_state_tables(const tbx_wrap *wrap, void *out_host, size_t cap, size_t *size);
/* Column j of snap_dev (uint32[rows][k]) <- env ids_dev[j] (ids_dev == NULL: env j).  Ids may repeat. */
int tbx_state_save(tbx_pool *pool, const int32_t *ids_dev, int k, uint32_t *snap_dev, void *stream);
/* Env ids_dev[j] <- column cols_dev[j] of snap_dev (uint32[rows][k_snap]), j < n; cols_dev == NULL: column j, ids_dev == NULL:
 * env j.  An env listed more than once receives the last listed column, whole.  When the blob's tables are byte-identical to
 * the pool's first table_count tables (always for the pool's own snapshots and for pools of the same config) table indices are
 * copied as they are; otherwise the blob's tables are added to the pool (this synchronises the device) and the indices
 * remapped, so snapshots move between pools, configs and GPUs of the same game.
 * Save and load enqueue all device work on `stream`; in the same-table case neither synchronises nor allocates after a pool's
 * first load, so save + load + step + render can be captured in a CUDA graph. */
int tbx_state_load(tbx_pool *pool, const uint32_t *snap_dev, int k_snap, const int32_t *cols_dev, const int32_t *ids_dev, int n,
                   const void *tables_blob, size_t blob_bytes, void *stream);
int tbx_wrap_state_save(tbx_wrap *wrap, const int32_t *ids_dev, int k, uint32_t *snap_dev, void *stream);
int tbx_wrap_state_load(tbx_wrap *wrap, const uint32_t *snap_dev, int k_snap, const int32_t *cols_dev, const int32_t *ids_dev, int n,
                        const void *tables_blob, size_t blob_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif
