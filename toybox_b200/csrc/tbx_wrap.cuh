/* tbx_wrap.cuh -- the DeepMind-style wrapper stack of baselines, fused into ONE thread-per-env kernel per agent step.
 *
 * Reference (baselines/baselines/common/atari_wrappers.py): make_atari = MaxAndSkipEnv(NoopResetEnv(env, 30), 4)
 * (:323-333), wrap_deepmind = FrameStack(ClipRewardEnv(WarpFrame(FireResetEnv(EpisodicLifeEnv(env)))), 4) (:345-360),
 * driven by a VecEnv worker that resets an env as soon as it reports done (vec_env/subproc_vec_env.py:11-15).
 * Per agent step the reference makes 4 ctoybox transitions + 4 full renders per env and keeps the pixel-wise max
 * of the last two frames; here one kernel runs the 4 transitions (and, for finished envs, the whole reset sequence
 * -- new_game, the random no-ops, the FIRE / RIGHT steps of FireResetEnv) and snapshots the state before the last
 * transition, so the render kernel (tbx_render_area.cuh, dual mode) needs to draw just the two states whose max
 * is the observation.  Frames that the reference renders and throws away are never drawn.
 *
 * Per-env wrapper state (5 words, word-major like the planes): EpisodicLifeEnv.lives, .was_real_done, the number of
 * NoopResetEnv resets so far (the counter of the no-op count generator), and the two accumulators of baselines' Monitor
 * (bench/monitor.py:58-76), which sits between make_atari and wrap_deepmind (common/cmd_util.py:30-36, run.py:116-119):
 * the sum of raw rewards and the number of MaxAndSkipEnv steps since the last real reset -- the FIRE / RIGHT steps of
 * FireResetEnv.reset and the NOOP step of a life-loss reset count, the no-op frames of NoopResetEnv (below Monitor) do not.
 *
 * Sticky actions (repeat_action_probability, Machado et al. 2018; ALE's `if (rand() >= p) m_player_a_action = action`),
 * the STICKY instantiation: a layer directly above ToyboxBaseEnv, so the rule holds on every game frame the stack runs --
 * the skipped frames of an agent step, the no-op frames of NoopResetEnv, the FIRE / RIGHT steps of FireResetEnv and the
 * NOOP step of a life-loss reset.  Each frame repeats the ALE id of the env's previous frame where the draw
 * tbx_sticky_draw(sticky_seed, env0 + i, f) < sticky_thr (= llround(p * 2^32)), else applies the requested id; f counts
 * the env's frames and is never reset, and new_game sets the remembered id to NOOP (ALE's reset_game).  Both are two more
 * wrapper words (7 per env).
 * Episode time limit (max_steps > 0; gym's TimeLimit inside make_atari, between MaxAndSkipEnv and Monitor): its step
 * count is Monitor's length, and it is tested at the end of the agent's own step.  An env at the limit reports done (so
 * EpisodicLifeEnv sees was_real_done and the full reset chain runs) and Monitor's record, and `truncated` where its game
 * is not over (gym's info['TimeLimit.truncated'] = not done).
 * Deviations, all stated in DESIGN.md: the no-op count comes from the counter-based generator of this library
 * (tbx_action_index) instead of gym's np_random (a MT19937 seeded through gym's hash_seed: not part of ctoybox); the
 * sticky draws come from the same kind of generator instead of ALE's MT19937; reset-chain steps that cross the time limit
 * truncate at the next agent step.
 */
#ifndef TBX_WRAP_CUH
#define TBX_WRAP_CUH
#include "tbx_render.cuh"

namespace tbxk {

struct WrapArgs {
  uint32_t *planes, *planes_prev; /* state after the agent step / before its last frame (max of the two = observation) */
  uint32_t *wstate;               /* [5][n_pad]: el_lives, was_real_done, resets, monitor return, monitor length;
                                     [7][n_pad] when STICKY: + the ALE id of the last frame, the frame counter */
  int n, n_pad;
  const void *cfg, *tables;
  const int32_t *legal; /* the game's legal ALE ids: gym action index -> ALE id (envs/atari/base.py:126) */
  int n_legal;
  const int32_t *actions; /* int32[N] gym action indices; NULL = reset every env (VecEnv.reset) */
  int skip, noop_max, episodic_life, fire_reset, clip_rewards;
  uint64_t noop_seed, env0;
  uint64_t sticky_seed, sticky_thr; /* STICKY: a frame repeats the last id where tbx_sticky_draw(sticky_seed, env0 + i, f) < sticky_thr */
  int max_steps;                    /* TimeLimit: 0 = none */
  int32_t *reward, *score, *lives; /* reward: summed over the skipped frames, sign() of it when clip_rewards */
  uint8_t *done, *real_done, *was_reset; /* done as the agent sees it; game over; observation comes from a reset */
  int32_t *ep_return, *ep_length; /* may be NULL: Monitor's {'r', 'l'} of the episode that ended in this agent step (where real_done or truncated) */
  uint8_t *truncated;             /* may be NULL: the agent step hit the time limit before the game was over */
  unsigned long long *stats;
  int *bad_actions;
};

/* The wrapper chain is a small state machine over UNITS of frames, so that the (large) transition and new_game code
 * is instantiated once: a unit is either one MaxAndSkipEnv.step (`skip` frames of one action, stops at game over,
 * snapshots the state before its last frame) or the no-op frames of NoopResetEnv.reset.  Stages name the caller a
 * finished unit returns to. */
enum { TBX_U_SKIP = 0, TBX_U_NOOP = 1 };
enum { TBX_ST_MAIN = 0, TBX_ST_ELR_A, TBX_ST_FIRE1, TBX_ST_ELR_B, TBX_ST_FIRE2, TBX_ST_ELR_C, TBX_ST_END };

template <int GAME, bool STICKY>
__global__ void __launch_bounds__(128) wrap_step_kernel(WrapArgs a) {
  typedef Traits<GAME> T;
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= a.n) return;
  const typename T::Cfg &cfg = *(const typename T::Cfg *)a.cfg;
  const typename T::Table *tables = (const typename T::Table *)a.tables;
  TbxAcc S;
  S.p = a.planes + env;
  S.stride = (size_t)a.n_pad;
  int el_lives = (int)a.wstate[env];                         /* EpisodicLifeEnv.lives */
  int was_real_done = (int)a.wstate[(size_t)a.n_pad + env];   /* EpisodicLifeEnv.was_real_done */
  int resets = (int)a.wstate[2 * (size_t)a.n_pad + env];      /* NoopResetEnv resets so far */
  int mon_ret = (int)a.wstate[3 * (size_t)a.n_pad + env];     /* Monitor.rewards: sum and count since Monitor.reset */
  int mon_len = (int)a.wstate[4 * (size_t)a.n_pad + env];
  int sticky_ale = 0;   /* STICKY: the ALE id applied on the env's last frame */
  uint32_t frame = 0;   /* STICKY: the env's frame counter, the draw's key */
  if (STICKY) {
    sticky_ale = (int)a.wstate[5 * (size_t)a.n_pad + env];
    frame = a.wstate[6 * (size_t)a.n_pad + env];
  }
  int unit_rew = 0, ep_ret_out = 0, ep_len_out = 0;

  int total = 0, sink = 0;
  bool out_done = false, out_real = false, out_trunc = false, reset = false;
  int stage = TBX_ST_END, unit = TBX_U_SKIP, frames_left = 0, ale = 0;
  bool snapped = false, unit_done = false, need_new_game = false;
  int score_out = S.ldi(TBX_HW(score)), lives_out = S.ldi(TBX_HW(lives));

#define TBX_SNAPSHOT() \
  do { for (int w_ = 0; w_ < T::RW; w_++) a.planes_prev[(size_t)w_ * a.n_pad + env] = a.planes[(size_t)w_ * a.n_pad + env]; } while (0)
  /* MaxAndSkipEnv.step(action) (atari_wrappers.py:189-206) */
#define TBX_START_SKIP(ALE) \
  do { unit = TBX_U_SKIP; ale = (ALE); frames_left = a.skip; snapped = false; unit_done = false; unit_rew = 0; } while (0)
  /* EpisodicLifeEnv.reset (:172-184): NoopResetEnv.reset (:120-134) after a real game over (always, without
   * EpisodicLifeEnv), else one NOOP agent step */
#define TBX_START_EL_RESET() \
  do { \
    if (!a.episodic_life || was_real_done) { \
      need_new_game = true; unit = TBX_U_NOOP; ale = a.legal[0]; unit_done = false; mon_ret = 0; mon_len = 0; /* Monitor.reset */ \
      frames_left = a.noop_max > 0 ? 1 + (int)tbx_action_index(a.noop_seed, a.env0 + (uint64_t)env, (uint64_t)resets, (uint32_t)a.noop_max) : 0; \
    } else TBX_START_SKIP(a.legal[0]); \
  } while (0)

  if (a.actions) {
    const int idx = a.actions[env];
    if (idx < 0 || idx >= a.n_legal) { atomicAdd(a.bad_actions, 1); TBX_SNAPSHOT(); }
    else { stage = TBX_ST_MAIN; TBX_START_SKIP(a.legal[idx]); }
  } else { /* VecEnv.reset(): the wrappers' reset chain (a new game only where the last game is over, as in the reference) */
    reset = true;
    stage = TBX_ST_ELR_A;
    TBX_START_EL_RESET();
  }

  while (stage != TBX_ST_END) {
    if (need_new_game) { /* ToyboxBaseEnv.reset (envs/atari/base.py:151-156) */
      T::new_game(S, cfg, tables);
      need_new_game = false;
      if (STICKY) sticky_ale = 0; /* ALE's reset_game: the remembered action is NOOP */
    }
    if (frames_left > 0) {
      if (unit == TBX_U_SKIP && frames_left == 1 && a.skip > 1) { TBX_SNAPSHOT(); snapped = true; } /* the state before the last repeat */
      /* ToyboxBaseEnv.step (base.py:115-149): one transition, reward = max(score - prev, 0), done = lives <= 0 */
      const int lives_before = S.ldi(TBX_HW(lives));
      int applied = ale;
      if (STICKY) { /* sticky actions: repeat the last frame's id with probability p */
        if ((uint64_t)tbx_sticky_draw(a.sticky_seed, a.env0 + (uint64_t)env, (uint64_t)frame) >= a.sticky_thr) sticky_ale = ale;
        frame++;
        applied = sticky_ale;
      }
      T::step(S, cfg, tables, tbx_ale_action_to_input(applied));
      const TbxStepOut o = tbx_bookkeep(S, lives_before);
      if (stage == TBX_ST_MAIN) total += o.reward; else sink += o.reward;
      unit_rew += o.reward;
      if (o.episode_ended) {
        atomicAdd(a.stats + 0, 1ull);
        atomicAdd(a.stats + 1, (unsigned long long)(long long)o.ep_return);
        atomicAdd(a.stats + 2, (unsigned long long)o.ep_len);
        atomicMax((long long *)(a.stats + 3), (long long)o.ep_return);
      }
      frames_left--;
      if (o.done) {
        if (unit == TBX_U_NOOP) need_new_game = true; /* NoopResetEnv: "if done: obs = self.env.reset()" */
        else { unit_done = true; frames_left = 0; }    /* MaxAndSkipEnv: "if done: break" */
      }
      if (frames_left > 0 || need_new_game) continue;
    }
    /* the unit is complete */
    if (unit == TBX_U_SKIP) { mon_ret += unit_rew; mon_len += 1; } /* Monitor.step above MaxAndSkipEnv */
    if (unit == TBX_U_NOOP) { resets++; TBX_SNAPSHOT(); }   /* the observation of a reset is a single frame */
    else if (!snapped) TBX_SNAPSHOT();                      /* stopped early: the reference's observation is stale and unused */
    bool done = unit_done;
    if (stage == TBX_ST_MAIN && a.max_steps > 0 && mon_len >= a.max_steps) { /* TimeLimit.step, on the agent's step only */
      out_trunc = !done; /* info['TimeLimit.truncated'] = not done */
      done = true;
    }
    if (stage == TBX_ST_MAIN || stage == TBX_ST_FIRE1 || stage == TBX_ST_FIRE2) {
      if (stage == TBX_ST_MAIN) { out_real = unit_done; if (done) { ep_ret_out = mon_ret; ep_len_out = mon_len; } } /* info['episode'] reaches the agent */
      if (a.episodic_life) { /* EpisodicLifeEnv.step (:158-170) */
        was_real_done = done;
        const int lives = S.ldi(TBX_HW(lives));
        if (lives < el_lives && lives > 0) done = true;
        el_lives = lives;
      }
    } else {
      el_lives = S.ldi(TBX_HW(lives)); /* end of EpisodicLifeEnv.reset */
    }
    switch (stage) {
      case TBX_ST_MAIN:
        out_done = done;
        score_out = S.ldi(TBX_HW(score)); lives_out = S.ldi(TBX_HW(lives));
        if (done) { reset = true; stage = TBX_ST_ELR_A; TBX_START_EL_RESET(); } /* the VecEnv worker resets a finished env at once */
        else stage = TBX_ST_END;
        break;
      case TBX_ST_ELR_A: /* FireResetEnv.reset (:143-152): reset, agent step FIRE (index 1), agent step index 2 */
        if (a.fire_reset && a.n_legal >= 3) { stage = TBX_ST_FIRE1; TBX_START_SKIP(a.legal[1]); }
        else stage = TBX_ST_END;
        break;
      case TBX_ST_FIRE1:
        if (done) { stage = TBX_ST_ELR_B; TBX_START_EL_RESET(); }
        else { stage = TBX_ST_FIRE2; TBX_START_SKIP(a.legal[2]); }
        break;
      case TBX_ST_ELR_B:
        stage = TBX_ST_FIRE2; TBX_START_SKIP(a.legal[2]);
        break;
      case TBX_ST_FIRE2:
        if (done) { stage = TBX_ST_ELR_C; TBX_START_EL_RESET(); }
        else stage = TBX_ST_END;
        break;
      default:
        stage = TBX_ST_END;
        break;
    }
  }
#undef TBX_SNAPSHOT
#undef TBX_START_SKIP
#undef TBX_START_EL_RESET

  a.wstate[env] = (uint32_t)el_lives;
  a.wstate[(size_t)a.n_pad + env] = (uint32_t)was_real_done;
  a.wstate[2 * (size_t)a.n_pad + env] = (uint32_t)resets;
  a.wstate[3 * (size_t)a.n_pad + env] = (uint32_t)mon_ret;
  a.wstate[4 * (size_t)a.n_pad + env] = (uint32_t)mon_len;
  if (STICKY) {
    a.wstate[5 * (size_t)a.n_pad + env] = (uint32_t)sticky_ale;
    a.wstate[6 * (size_t)a.n_pad + env] = frame;
  }
  if (a.ep_return) a.ep_return[env] = ep_ret_out;
  if (a.ep_length) a.ep_length[env] = ep_len_out;
  if (a.reward) a.reward[env] = a.clip_rewards ? (total > 0 ? 1 : total < 0 ? -1 : 0) : total;
  if (a.done) a.done[env] = (uint8_t)out_done;
  if (a.real_done) a.real_done[env] = (uint8_t)out_real;
  if (a.was_reset) a.was_reset[env] = (uint8_t)reset;
  if (a.truncated) a.truncated[env] = (uint8_t)out_trunc;
  if (a.score) a.score[env] = score_out;
  if (a.lives) a.lives[env] = lives_out;
}

} /* namespace tbxk */
#endif
