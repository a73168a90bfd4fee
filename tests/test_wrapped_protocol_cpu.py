"""CPU tier: the checker of sticky actions and the episode time limit of the fused wrapper stack (DESIGN.md 4.5) --
tests/wrapped_protocol_ref.py: StickyActionEnv (ALE's repeat_action_probability, directly above the base env), TimeLimit (gym's
TimeLimit between MaxAndSkipEnv and Monitor) and ProtocolWrappedEnv, the oracle-side wrapper chain with both, which
tests/test_gpu_wrapped_protocol.py compares the GPU with.

Checked here: the sticky draw is the upper half of the oracle's splitmix64 mix keyed by the salted seed; the rule's counts
follow the binomial law and its extremes (p = 0 never, p = 1 always sticky); the chain with both features off computes what
WrappedEnv computed before they existed (committed trajectory digests); at p = 1 Breakout's paddle never moves; truncated
episodes end at the limit, or up to the length of a life-loss reset chain past it, are flagged and take the full reset chain,
and a game over on the limit step is a game over, not a truncation."""
import hashlib

import numpy as np
import pytest

import wrapped_protocol_ref as R


def test_sticky_draw_is_the_stated_formula(oracle_mod):
    """u = upper 32 bits of mix(seed ^ salt, env, f): oracle/common.c's action index of that mix, reduced to n = 2^31 and
    n = 2^32 - 1, fixes all 32 bits"""
    O = oracle_mod
    rng = np.random.default_rng(5)
    keys = [(int(s), int(e), int(f)) for s, e, f in zip(rng.integers(0, 1 << 63, 300, dtype=np.int64) * 2 + 1,
                                                        rng.integers(0, 1 << 20, 300), rng.integers(0, 1 << 40, 300))]
    keys += [(0, 0, 0), (R.M64, R.M64, R.M64), (R.STICKY_SALT, 0, 0), (7, 3, 1 << 32)]
    for s, e, f in keys:
        u = R.sticky_draw(s, e, f)
        for n in (1 << 31, (1 << 32) - 1, 30):
            assert O.action_index(s ^ R.STICKY_SALT, e, f, n) == (u * n) >> 32, (s, e, f, n)
    # one seed for both streams: the sticky draws are not the no-op stream's numbers
    same = sum(R.sticky_draw(9, e, f) == R.mix(9, e, f) >> 32 for e in range(4) for f in range(500))
    assert same == 0
    assert [R.sticky_threshold(p) for p in (0.0, 0.25, 1.0, 2.0 ** -33)] == [0, 1 << 30, 1 << 32, 1]   # llround, halves away


class _Recorder:
    """a base env that records the ALE ids it is stepped with"""
    legal = [0, 1, 3, 4]

    def __init__(self):
        self.applied = []

    def step(self, a):
        self.applied.append(self.legal[a])
        return None, 0, False, {}

    def reset(self):
        return None


@pytest.mark.parametrize("p", [0.1, 0.25, 0.9])
def test_sticky_counts_within_binomial_bounds(oracle_mod, p):
    n, seed, env_id = 100_000, 0x51C4, 11
    base = _Recorder()
    env = R.StickyActionEnv(base, p, seed, env_id)
    requested = [(f * 7 + f // 3) % 4 for f in range(n)]          # the request changes on most frames
    for a in requested:
        env.step(a)
    thr = R.sticky_threshold(p)
    sticky = [R.sticky_draw(seed, env_id, f) < thr for f in range(n)]
    want, prev = [], 0
    for f in range(n):
        if not sticky[f]:
            prev = base.legal[requested[f]]
        want.append(prev)
    assert base.applied == want                                    # the rule, frame by frame
    k = sum(sticky)
    sd = (n * p * (1 - p)) ** 0.5
    assert abs(k - n * p) < 5 * sd, (k, n * p, sd)
    assert env.f == n


def test_sticky_extremes(oracle_mod):
    for p, applied in ((0.0, None), (1.0, 0)):
        base = _Recorder()
        env = R.StickyActionEnv(base, p, 3, 0)
        env.prev = 3 if p == 1.0 else 0
        env.reset()                                                # new_game remembers NOOP
        for f in range(20_000):
            env.step(1 + f % 3)
        if applied is None:
            assert base.applied == [base.legal[1 + f % 3] for f in range(20_000)]
        else:
            assert set(base.applied) == {applied}


# sha256 of oracle.wrappers.WrappedEnv's trajectories in _digest, recorded before sticky actions and the time limit existed
DIGESTS = [
    ("breakout", {}, "6ec4ff19ba80021ab61dfcd8fac483c28db9fe3e85e0ee927d849980b4f15071"),
    ("amidar", {}, "d247e2950460710e85a4e6d11ae1068006ab1724d15c4cff9a06e285b272b9e5"),
    ("space_invaders", {}, "e3cb604a8232f2dd870c8feaa85f847ca6e36a74466b98ffe74b0dca07c6617f"),
    ("breakout", dict(frame_skip=3, noop_max=0, episode_life=False, stack_reset="zero"),
     "12d6a8c5741ce1d299fbab5f7f782df543cba35cd5bf21120c08a4e05487dc46"),
]


def _digest(O, cls, game, kw, steps=120):
    env = cls(game, 21, env_id=3, noop_seed=4, **kw)
    h = hashlib.sha256(env.reset().tobytes())
    n = len(env.base.legal)
    for t in range(steps):
        obs, r, d, info = env.step(O.action_index(0xB200, 3, t, n))
        assert not info.get("truncated")
        h.update(obs.tobytes())
        ep = info.get("episode", {})
        h.update(repr((r, d, info["score"], info["lives"], info["real_done"], info["fresh"], ep.get("r"), ep.get("l"))).encode())
    return h.hexdigest()


@pytest.mark.parametrize("game,kw,digest", DIGESTS)
def test_defaults_leave_the_chain_as_it_was(oracle_mod, game, kw, digest):
    from oracle import wrappers as OW
    assert _digest(oracle_mod, OW.WrappedEnv, game, kw) == digest
    assert _digest(oracle_mod, R.ProtocolWrappedEnv, game, kw) == digest
    assert _digest(oracle_mod, R.ProtocolWrappedEnv, game, dict(kw, repeat_action_probability=0.0, max_episode_steps=0)) == digest


def test_always_sticky_breakout_paddle_stays_put(oracle_mod):
    """p = 1: every frame repeats the last one, and a new game remembers NOOP, so no requested action ever takes effect"""
    from oracle import wrappers as OW
    env = R.ProtocolWrappedEnv("breakout", 8, env_id=1, noop_seed=2, repeat_action_probability=1.0)
    env.reset()
    x0 = env.base.b.states[0].paddle.position.x
    for t in range(150):
        env.step(2 + t % 2)                                        # RIGHT / LEFT, never NOOP
        assert env.base.b.states[0].paddle.position.x == x0, t
    free = OW.WrappedEnv("breakout", 8, env_id=1, noop_seed=2)
    free.reset()
    for t in range(10):
        free.step(2)
    assert free.base.b.states[0].paddle.position.x != x0           # the same actions do move it without stickiness


def _limit_run(O, L, steps, kw, seed=31, lives=None):
    env = R.ProtocolWrappedEnv("breakout", seed, env_id=0, noop_seed=6, max_episode_steps=L, **kw)
    env.reset()
    if lives is not None:                                          # a short game: the first lost ball ends it
        js = env.base.b.state_json(0)
        js["lives"] = lives
        env.base.b.write_state_json(0, js)
    n = len(env.base.legal)
    out = []
    for t in range(steps):
        obs, r, d, info = env.step(O.action_index(0xB1, 0, t, n))
        out.append((d, info, env.base.lives(), len(env.monitor.rewards)))
    return out


@pytest.mark.parametrize("kw", [{}, dict(repeat_action_probability=0.25)])
def test_time_limit_truncates_and_resets(oracle_mod, kw):
    L = 37
    run = _limit_run(oracle_mod, L, 700, kw)
    ntrunc = 0
    for t, (d, info, lives_after, len_after) in enumerate(run):
        if info["truncated"]:
            ntrunc += 1
            assert d and not info["real_done"] and "episode" in info, t
            # the limit is tested on the agent's step: its own step reaches L, or the reset chain of a lost life in the step
            # before (EpisodicLifeEnv's NOOP, FireResetEnv's FIRE and RIGHT: 3 steps) carried the count past it
            l = info["episode"]["l"]
            assert L <= l <= L + 3, (t, l)
            if l > L:
                pd, pinfo = run[t - 1][:2]
                assert pd and not pinfo["real_done"] and not pinfo["truncated"], (t, l)
            # the full reset chain: a new game, and Monitor restarted with FireResetEnv's two steps
            assert lives_after == 5 and len_after == 2, (t, lives_after, len_after)
        elif "episode" in info:
            assert info["real_done"], t
        if not d:
            assert len_after < L, t                               # no agent step ends at or past the limit untruncated
    assert ntrunc >= 10, ntrunc


def test_reset_chain_crossing_the_limit_truncates_at_the_next_agent_step(oracle_mod):
    """a life lost one step short of the limit: its reset chain (NOOP, FIRE, RIGHT) carries Monitor's count past the limit,
    and the next agent step truncates with l = L + 3 (DESIGN.md 4.5)"""
    O = oracle_mod
    free = _limit_run(O, 0, 400, {})
    t = next(t for t, (d, info, *_) in enumerate(free) if d and not info["real_done"])   # the first lost life
    L = free[t][3] - 3 + 1                                         # Monitor's count after that agent step, plus one
    capped = _limit_run(O, L, t + 2, {})
    assert not any(x[1]["truncated"] for x in capped[:t + 1])
    d, info = capped[t + 1][:2]
    assert d and info["truncated"] and info["episode"]["l"] == L + 3


def test_game_over_on_the_limit_step_is_not_truncated(oracle_mod):
    O = oracle_mod
    free = _limit_run(O, 0, 400, {}, lives=1)                  # 0: no limit
    ends = [t for t, (d, info, *_) in enumerate(free) if info["real_done"]]
    assert ends, "the one-life game ends"
    L = free[ends[0]][1]["episode"]["l"]                           # the game ends on its L-th step
    capped = _limit_run(O, L, ends[0] + 1, {}, lives=1)
    d, info = capped[-1][:2]
    assert d and info["real_done"] and not info["truncated"] and info["episode"]["l"] == L
    assert not any(x[1]["truncated"] for x in capped)
