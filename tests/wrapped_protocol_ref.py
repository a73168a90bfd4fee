"""TEST INFRASTRUCTURE: the checker for sticky actions and the episode time limit of the fused wrapper stack
(DeepmindToybox(repeat_action_probability, sticky_seed, max_episode_steps); DESIGN.md 4.5).  It extends the oracle-side
wrapper chain (oracle/wrappers.py, left as it is) with two layers, each a restatement of the reference behaviour it follows:

  StickyActionEnv  ALE's sticky actions (repeat_action_probability; Machado et al. 2018; ALE v5 defaults to p = 0.25), directly
                   above the base env, so it acts on every game frame: skipped frames, NoopResetEnv's no-ops, FireResetEnv's
                   FIRE / index-2 steps and the NOOP step of a life-loss reset.  Frame f of env i repeats the ALE id of the
                   env's previous frame where u < thr (ALE: `if (rand() >= p) m_player_a_action = action`), else applies the
                   requested id; u = sticky_draw(sticky_seed, env0 + i, f), thr = llround(p * 2^32), so p = 0 is never and
                   p = 1 always sticky; f counts the env's frames and is never reset; a new game remembers NOOP (ALE's
                   reset_game).  The counter-based draw replaces ALE's MT19937.
  TimeLimit        gym's TimeLimit as baselines' make_atari(env_id, max_episode_steps) places it, between MaxAndSkipEnv and
                   Monitor, so its count is Monitor's episode length.  It truncates only on the agent's own step (armed by
                   ProtocolWrappedEnv.step): done is set, so EpisodicLifeEnv sees was_real_done and the full reset chain
                   runs, Monitor reports the episode, and info['TimeLimit.truncated'] = not done (game over).  Reset-chain
                   steps that cross the limit truncate at the next agent step.

ProtocolWrappedEnv is oracle.wrappers.WrappedEnv with both layers in place; its step() info gains 'truncated'.  With p = 0 and
no limit it builds exactly WrappedEnv's chain."""
import math

import numpy as np

from oracle import oracle as O
from oracle import wrappers as OW

M64 = (1 << 64) - 1
STICKY_SALT = 0x5354494B59414354        # "STIKYACT": separates the sticky draws from the no-op draws of the same seed


def mix(seed, env, t):
    """the splitmix64 finaliser of (seed, env, t) that keys the library's counter-based streams (tbx_common.h:tbx_mix;
    oracle/common.c:tbo_action_index reduces its upper 32 bits to an action index)"""
    z = (seed + env * 0x9E3779B97F4A7C15 + t * 0xD1B54A32D192ED03) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def sticky_draw(seed, env, f):
    """the sticky-action draw of env `env` on its frame `f`: uniform over [0, 2^32)"""
    return mix((seed ^ STICKY_SALT) & M64, env, f) >> 32


def sticky_threshold(p):
    """llround(p * 2^32): p * 2^32 and the + 0.5 are exact in f64 below 2^52"""
    return math.floor(p * 2 ** 32 + 0.5)


class StickyActionEnv:
    def __init__(self, env, p, seed, env_id):
        self.env, self.seed, self.env_id = env, seed, env_id
        self.thr = sticky_threshold(p)
        self.prev, self.f = 0, 0                         # ALE id of the last frame (NOOP), frame counter
        self.legal = env.legal

    def step(self, action_index):
        if not sticky_draw(self.seed, self.env_id, self.f) < self.thr:
            self.prev = self.legal[action_index]
        self.f += 1
        return self.env.step(self.legal.index(self.prev))

    def reset(self):
        self.prev = 0
        return self.env.reset()


class TimeLimit:                                        # gym/wrappers/time_limit.py
    def __init__(self, env, max_episode_steps):
        self.env, self.max, self.elapsed, self.armed = env, max_episode_steps, 0, False

    def step(self, ac):
        ob, rew, done, info = self.env.step(ac)
        self.elapsed += 1
        armed, self.armed = self.armed, False
        if armed and self.elapsed >= self.max:
            info = dict(info)
            info["TimeLimit.truncated"] = not done
            done = True
        return ob, rew, done, info

    def reset(self):
        self.elapsed = 0
        return self.env.reset()


class ProtocolWrappedEnv(OW.WrappedEnv):
    """OW.WrappedEnv(game, seed, ...) with StickyActionEnv under NoopResetEnv (repeat_action_probability > 0; sticky_seed
    defaults to noop_seed) and TimeLimit between MaxAndSkipEnv and Monitor (max_episode_steps > 0)"""

    def __init__(self, game, seed, env_id=0, frame_skip=4, noop_max=30, episode_life=True, fire_reset=True, clip_rewards=True,
                 frame_stack=4, size=(84, 84), noop_seed=0, stack_reset="fill", repeat_action_probability=0.0, sticky_seed=None,
                 max_episode_steps=None):
        super().__init__(game, seed, env_id=env_id, frame_skip=frame_skip, noop_max=noop_max, episode_life=episode_life,
                         fire_reset=fire_reset, clip_rewards=clip_rewards, frame_stack=frame_stack, size=size, noop_seed=noop_seed,
                         stack_reset=stack_reset)
        # rebuild the chain below EpisodicLifeEnv with the two layers (the same classes and order as WrappedEnv.__init__)
        dims = O.DIMS[game]
        env = self.base
        if repeat_action_probability > 0:
            env = StickyActionEnv(env, repeat_action_probability, noop_seed if sticky_seed is None else sticky_seed, env_id)
        env = OW.NoopResetEnv(env, noop_max, noop_seed, env_id) if noop_max > 0 else OW._PlainReset(env)
        self.skipper = env = OW.MaxAndSkipEnv(env, frame_skip, (dims[1], dims[0]))
        self.limit = None
        if max_episode_steps:
            self.limit = env = TimeLimit(env, max_episode_steps)
        self.monitor = env = OW.Monitor(env)
        if episode_life:
            env = OW.EpisodicLifeEnv(env, self.base)
        if fire_reset and len(self.base.legal) >= 3:
            env = OW.FireResetEnv(env)
        self.env = self._top = _InfoTap(env)

    def step(self, action):
        if self.limit is not None:
            self.limit.armed = True
        stacked, reward, done, out = super().step(action)
        out["truncated"] = bool(self._top.info.get("TimeLimit.truncated", False))
        return stacked, reward, done, out


class _InfoTap:
    """the top of the chain: passes steps and resets through and keeps the info of the last step, which WrappedEnv.step
    reduces to its own fields"""

    def __init__(self, env):
        self.env, self.info = env, {}

    def step(self, ac):
        ob, rew, done, self.info = self.env.step(ac)
        return ob, rew, done, self.info

    def reset(self):
        return self.env.reset()


def colour(env, size):
    """env with WarpFrame(grayscale=False), as test_wrapped_rgb_cpu.colour_wrapped_env builds it"""
    from test_rgb_area_cpu import rgb_area
    env._warp = lambda obs: rgb_area(O, obs, size[0], size[1])
    base = env.base
    base._obs = lambda: base.b.render("rgb")[0]
    env.skipper._obs_buffer = np.zeros(env.skipper._obs_buffer.shape + (3,), np.uint8)
    return env
