"""TEST INFRASTRUCTURE: the checker for the final observations of the fused wrapper stack (DeepmindToybox(final_observation=True),
tbx_wrap_set_final_observations; DESIGN.md 4.5).  FinalObsEnv is wrapped_protocol_ref.ProtocolWrappedEnv (left as it is) with
two taps:

  the final stack  np.stack(self.frames) at the moment the VecEnv worker resets a finished env, i.e. the FrameStack the
                   reference held just before reset(): the k-1 newest frames before the step and WarpFrame of the
                   MaxAndSkipEnv.step observation of this step -- under both stack modes;
  the stop index   the frame index at which the agent's own MaxAndSkipEnv.step stopped (skip-1 for a full step, less where
                   the game ended early and the buffer's max shows stale slots), and the observations of its last two
                   frames, so that tests can show where the stale slots make a difference.

step() info gains 'final' (the [k, h, w(, 3)] stack, or None when the step did not end in done), 'stop' and 'last2'."""
import numpy as np

import wrapped_protocol_ref as R


class _FrameTap:
    """sits between MaxAndSkipEnv and the env below it: counts the frames of the current MaxAndSkipEnv.step and keeps the
    last two observations"""

    def __init__(self, env):
        self.env, self.n, self.last = env, 0, []

    def step(self, ac):
        out = self.env.step(ac)
        self.n += 1
        self.last = (self.last + [out[0].copy()])[-2:]
        return out

    def reset(self):
        return self.env.reset()

    def __getattr__(self, name):
        return getattr(self.env, name)


class FinalObsEnv(R.ProtocolWrappedEnv):
    def __init__(self, game, seed, **kw):
        super().__init__(game, seed, **kw)
        sk = self.skipper
        self.tap = sk.env = _FrameTap(sk.env)
        inner = sk.step

        def step(action):
            self.tap.n, self.tap.last = 0, []
            return inner(action)

        sk.step = step
        self._in_step, self._final, self._stop, self._last2 = False, None, None, None

    def reset(self):
        if self._in_step:       # the worker's reset of a finished env: the agent's MaxAndSkipEnv.step was the last one
            self._final = np.stack(self.frames)
            self._stop, self._last2 = self.tap.n - 1, list(self.tap.last)
        return super().reset()

    def step(self, action):
        self._in_step, self._final = True, None
        try:
            stacked, reward, done, out = super().step(action)
        finally:
            self._in_step = False
        if not done:
            self._stop, self._last2 = self.tap.n - 1, list(self.tap.last)
        out["final"], out["stop"], out["last2"] = self._final, self._stop, self._last2
        return stacked, reward, done, out


def one_life(js, i):
    """one life left in every env: random play then ends whole games"""
    js["lives"] = 1


def breakout_stagger(js, i):
    """Breakout, one life and a ball in flight away from the paddle, at a height and speed that differ per env: the games
    end on different frames of a MaxAndSkipEnv step (served balls all fall in step with each other)"""
    js.update(lives=1, is_dead=False, reset=False)
    js["balls"] = [{"position": {"x": 30.0 + 5 * (i % 5), "y": 100.0 + 3.0 * (i % 7)}, "velocity": {"x": 0.0, "y": 1.0 + 0.25 * (i % 8)}}]
    js["paddle"]["position"]["x"] = 200.0
