"""GPU tier: colour observations of the fused wrapper stack -- DeepmindToybox(grayscale=False) / ToyboxVecEnv(grayscale=False),
tbx_wrap_step under TBX_OBS_RGB_AREA, rendered by the dual RGB tile kernel -- env by env and bit for bit against the oracle-side
chain with WarpFrame(grayscale=False) (test_wrapped_rgb_cpu.colour_wrapped_env): the whole ring in FrameStack order, rewards,
dones, real dones, lives, scores and Monitor's episode records.

Covered: rollouts of the three games under both stack-reset modes with full game overs; the dual list sweep, per-tile rebuild
and both-frames flag at every D_SIZES size on adversarial states; configs whose colours share a gray; the wrapper switches; a
gray wrapped env stepping beside a colour one; the sizes and calls the colour stack refuses; the VecEnv surface; snapshots."""
import numpy as np
import pytest

from test_gpu_area_coverage import D_SIZES, D_VARIANTS, _assert_same, _intervene, _set
from test_gpu_rgb_area import _ami_twin_cfg, _brk_twin_cfg
from test_wrapped_rgb_cpu import colour_wrapped_env

pytestmark = pytest.mark.gpu
GAMES = ["breakout", "amidar", "space_invaders"]


def _flat(a, n):
    """a ring [n, k, h, w] or [n, k, h, w, 3] -> [n, k * h, w * channels] for _assert_same"""
    return a.reshape(n, -1, a.shape[-2] * a.shape[-1]) if a.ndim == 5 else a.reshape(n, -1, a.shape[-1])


def _last_life(js, i, rng):
    """one life left in every other env: Breakout's random play then ends whole games (real_done, Monitor records, full resets)"""
    if i % 2 == 0:
        js["lives"] = 1


class _Pair:
    """a DeepmindToybox and its per-env references, stepped together and compared after every step"""

    def __init__(self, game, n, kw, seed0=500, grayscale=False, config=None):
        import torch
        from oracle import wrappers as OW
        from toybox_b200.wrappers import DeepmindToybox
        self.torch, self.game, self.n = torch, game, n
        self.env = DeepmindToybox(game, n, seeds=seed0, noop_seed=7, grayscale=grayscale, config=config, **kw)
        if grayscale:
            self.refs = [OW.WrappedEnv(game, seed0 + i, env_id=i, noop_seed=7, **kw) for i in range(n)]
        else:
            self.refs = [colour_wrapped_env(game, seed0 + i, env_id=i, noop_seed=7, config=config, **kw) for i in range(n)]
        self.ndone = self.nreal = 0
        obs = self.env.reset()
        want = np.stack([r.reset() for r in self.refs])
        _assert_same(_flat(obs[:, self.env.order()].cpu().numpy(), n), _flat(want, n), "%s reset" % game)

    def edit(self, fn, rng):
        """the same state edit on both sides"""
        states = []
        for i, r in enumerate(self.refs):
            js = r.base.b.state_json(0)
            fn(js, i, rng)
            r.base.b.write_state_json(0, js)
            states.append(js)
        self.env.pool.write_state_json(states)

    def step(self, acts, what):
        env, n = self.env, self.n
        obs, rew, done, info = env.step(self.torch.as_tensor(acts, device=env.device))
        got = obs[:, env.order()].cpu().numpy()
        rew, done = rew.cpu().numpy(), done.cpu().numpy().astype(bool)
        lives, score, real = info["lives"].cpu().numpy(), info["score"].cpu().numpy(), info["real_done"].cpu().numpy().astype(bool)
        ep_r, ep_l = info["ep_return"].cpu().numpy(), info["ep_length"].cpu().numpy()
        wants = []
        for i, r in enumerate(self.refs):
            w_obs, w_rew, w_done, w_info = r.step(int(acts[i]))
            assert (w_rew, w_done, w_info["lives"], w_info["score"], w_info["real_done"]) == (rew[i], done[i], lives[i], score[i], real[i]), \
                (what, i, w_rew, rew[i], w_done, done[i], w_info, lives[i], score[i], real[i])
            assert ("episode" in w_info) == bool(real[i]), (what, i)
            if real[i]:
                assert (w_info["episode"]["r"], w_info["episode"]["l"]) == (ep_r[i], ep_l[i]), (what, i, w_info["episode"], ep_r[i], ep_l[i])
                self.nreal += 1
            self.ndone += int(w_done)
            wants.append(w_obs)
        _assert_same(_flat(got, n), _flat(np.stack(wants), n), what)

    def close(self):
        self.env.check()
        self.env.close()


def _acts(n, n_act, t):
    from oracle import oracle as O
    return np.asarray([O.action_index(0xB200, i, t, n_act) for i in range(n)], np.int32)


def _run(game, n, steps, kw, seed0=500, edits=(), variants=None, config=None):
    """edits: (agent step, fn(js, i, rng)) written into both sides before that step; variants: test switches cycled every 2 steps"""
    p = _Pair(game, n, kw, seed0, config=config)
    rng = np.random.default_rng(seed0)
    try:
        for t in range(steps):
            for at, fn in edits:
                if t == at:
                    p.edit(fn, rng)
            v = variants[(t // 2) % len(variants)] if variants else {}
            _set(v)
            p.step(_acts(n, p.env.n_actions, t), "%s %s step %d %s" % (game, kw, t, v))
    finally:
        _set({})
        p.close()
    return p


# -------------------------------------------------------------------------------------------------------- 1. rollouts
@pytest.mark.parametrize("stack_reset", ["fill", "zero"])
@pytest.mark.parametrize("game", GAMES)
def test_wrapped_rgb_rollout_bit_exact(game, stack_reset):
    if game == "breakout":
        p = _run(game, 8, 260, dict(stack_reset=stack_reset), edits=[(2, _last_life)])
        assert p.ndone > p.nreal > 0, (p.ndone, p.nreal)   # lost lives (EpisodicLife resets) and whole games (full resets)
    else:
        _run(game, 6, 90, dict(stack_reset=stack_reset))


# ------------------------------------------------------------------------------------------------------ 2. dual paths
@pytest.mark.parametrize("game", GAMES)
def test_wrapped_rgb_dual_paths(game):
    """every D_SIZES size, adversarial states written into both sides after three steps, the list capacity cycling through 3
    (per-tile rebuild), 24 (sweeps) and the default: the dual list sweep, the rebuild and the both-frames flag of every run,
    each once per channel with both windows"""
    for k, size in enumerate(D_SIZES[game]):
        _run(game, 6, 24, dict(size=size), seed0=600 + 10 * k, edits=[(3, lambda js, i, rng: _intervene(game, js, i, rng))],
             variants=D_VARIANTS)


# ------------------------------------------------------------------------------------------ 3. colours sharing a gray
def _brk_twin_edit(js, i, rng):
    for k in rng.choice(len(js["bricks"]), size=int(rng.integers(0, 60)), replace=False):
        js["bricks"][int(k)]["alive"] = False
    if i % 3 == 1:                   # the ball over the paddle: the two colours of one gray side by side
        js["balls"] = [{"position": {"x": js["paddle"]["position"]["x"], "y": 140.0}, "velocity": {"x": 1.0, "y": 1.0}}]


def _ami_paint_edit(js, i, rng):
    tiles = js["board"]["tiles"]
    for _ in range(4 + i):
        ty, tx, ln = int(rng.integers(31)), int(rng.integers(32)), int(rng.integers(1, 20))
        for k in range(ln):
            if tx + k < 32 and tiles[ty][tx + k] in ("Unpainted", "ChaseMarker"):
                tiles[ty][tx + k] = "Painted"


@pytest.mark.parametrize("game", ["breakout", "amidar"])
def test_wrapped_rgb_colours_sharing_a_gray(game):
    """configs whose colours differ in RGB and share a gray (Breakout brick rows in twin pairs, paddle and ball twins; Amidar's
    painted track a twin of the unpainted one, enemies a third colour of that gray), with states edited on both sides, under the
    default list and the per-tile rebuild.  A gray byte used in place of a colour shows as a wrong channel here.

    The both-frames merge with two colours of one gray (a primitive in place in both frames whose colour changes) cannot be
    reached through the wrapper: a slot's colour is fixed by the config and the slot's kind in all three games -- bricks by
    row, paddle, ball, player, enemies (Amidar enemies have one colour in every mode), HUD digits -- except Amidar's delta tile
    runs, whose colour follows their look.  A run keeps its extent only while its look stays, because painting a tile splits
    or grows the painted run it joins, and a tile's look changes only by painting; Space Invaders' laser colours are set when
    a laser appears and a laser moves every frame."""
    if game == "breakout":
        cfg, edit = _brk_twin_cfg(), _brk_twin_edit
    else:
        cfg, edit = _ami_twin_cfg(), _ami_paint_edit
    for k, size in enumerate([(84, 84), (64, 64)] if game == "breakout" else [(84, 84), (96, 80)]):
        _run(game, 8, 40, dict(size=size), seed0=40 + k, edits=[(2, edit), (20, edit)], variants=[{}, {"TBX_AREA_LCAP": "3"}], config=cfg)


# ----------------------------------------------------------------------------------------------------------- 4. switches
def test_wrapped_rgb_switches():
    _run("breakout", 6, 100, dict(frame_skip=2, noop_max=5, episode_life=False, fire_reset=False, clip_rewards=False, frame_stack=3, size=(64, 72)))
    _run("breakout", 6, 100, dict(frame_skip=1, noop_max=0, frame_stack=1))
    _run("amidar", 4, 50, dict(frame_skip=3, noop_max=0, clip_rewards=False, frame_stack=1))
    _run("space_invaders", 4, 50, dict(frame_skip=3, noop_max=3, frame_stack=3, episode_life=False, fire_reset=False))


# ------------------------------------------------------------------------------------------- 5. gray beside colour
@pytest.mark.parametrize("game", GAMES)
def test_gray_wrapped_unchanged_beside_colour(game):
    """a gray and a colour DeepmindToybox of the same game and seeds in one process, stepped alternately: each matches its own
    reference (the per-size render caches hold both layouts side by side)"""
    n = 5
    gray = _Pair(game, n, {}, 70, grayscale=True)
    col = _Pair(game, n, {}, 70)
    try:
        for t in range(60):
            acts = _acts(n, gray.env.n_actions, t)
            gray.step(acts, "%s gray step %d" % (game, t))
            col.step(acts, "%s colour step %d" % (game, t))
    finally:
        gray.close()
        col.close()


# ------------------------------------------------------------------------------------------------------------ 6. refusals
def _outcome(game, size, grayscale):
    from toybox_b200.wrappers import DeepmindToybox
    env = None
    try:
        env = DeepmindToybox(game, 2, seeds=1, size=size, grayscale=grayscale)
        env.reset()
        return "ok"
    except Exception as e:
        return "%s: %s" % (type(e).__name__, e)
    finally:
        if env is not None:
            env.close()


@pytest.mark.parametrize("game", GAMES)
def test_wrapped_rgb_refuses_what_gray_refuses(game):
    """over a sweep of sizes, the colour stack accepts a size exactly when the gray stack does, and refuses it with the same
    message (Breakout 100 x 37, Amidar and Space Invaders 64 x 64: more than 5 x 4 taps)"""
    must_refuse = {"breakout": [(100, 37)], "amidar": [(64, 64)], "space_invaders": [(64, 64)]}[game]
    n_ok = 0
    for size in must_refuse + [(w, h) for w in (23, 48, 64, 84, 100, 128) for h in (20, 37, 60, 84, 105, 128)]:
        gray, col = _outcome(game, size, True), _outcome(game, size, False)
        assert gray == col, (game, size, gray, col)
        if size in must_refuse:
            assert "wrapped observations need an output size" in gray, (game, size, gray)
        n_ok += gray == "ok"
    assert 0 < n_ok < 37, n_ok


def test_set_obs_mode_refusals():
    import ctypes as C
    from toybox_b200 import _lib
    from toybox_b200.wrappers import DeepmindToybox
    env = DeepmindToybox("breakout", 2, seeds=1)
    L = env.L
    try:
        for mode in (0, 1, 2, 5, -1):
            assert L.tbx_wrap_set_obs_mode(env._w, mode) == 1, mode                 # TBX_EINVAL
        assert b"observation layout" in L.tbx_last_error()
        assert L.tbx_wrap_set_obs_mode(env._w, 4) == 0 and L.tbx_wrap_set_obs_mode(env._w, 3) == 0   # before the first step
        env.reset()
        for mode in (3, 4):
            assert L.tbx_wrap_set_obs_mode(env._w, mode) == 1, mode
        assert b"before the first tbx_wrap_step" in L.tbx_last_error()
        assert L.tbx_wrap_set_obs_mode(None, 4) == 1
    finally:
        env.close()
    assert _lib.SIGNATURES["tbx_wrap_set_obs_mode"] == (C.c_int, [C.c_void_p, C.c_int])


# ------------------------------------------------------------------------------------------------------------- 7. VecEnv
def test_vec_env_rgb():
    """ToyboxVecEnv(grayscale=False): (N, 84, 84, 12) observations, frame-major channels, against the colour chain under
    VecFrameStack (a finished env's first 9 channels are zero, its last 3 the reset observation) with Monitor's records"""
    from toybox_b200.wrappers import ToyboxVecEnv
    n = 8
    venv = ToyboxVecEnv("breakout", n, seeds=40, noop_seed=9, grayscale=False)
    refs = [colour_wrapped_env("breakout", 40 + i, env_id=i, noop_seed=9, stack_reset="zero") for i in range(n)]

    def cat(frames):                 # [k, h, w, 3] -> [h, w, 3k], oldest frame's channels first
        return np.concatenate(list(frames), axis=-1)
    try:
        assert venv.observation_space.shape == (84, 84, 12) and venv.action_space.n == 4
        obs = venv.reset()
        assert obs.shape == (n, 84, 84, 12) and obs.dtype == np.uint8
        assert np.array_equal(obs, np.stack([cat(r.reset()) for r in refs]))
        rng = np.random.default_rng(1)
        states = []
        for i, r in enumerate(refs):
            js = r.base.b.state_json(0)
            _last_life(js, i, rng)
            r.base.b.write_state_json(0, js)
            states.append(js)
        venv.env.pool.write_state_json(states)
        episodes = finished = 0
        for t in range(260):
            acts = _acts(n, 4, t)
            obs, rew, done, infos = venv.step(acts)
            assert obs.shape == (n, 84, 84, 12) and len(infos) == n
            for i, r in enumerate(refs):
                w_obs, w_rew, w_done, w_info = r.step(int(acts[i]))
                assert np.array_equal(obs[i], cat(w_obs)) and w_rew == rew[i] and w_done == done[i], (t, i)
                assert ("episode" in infos[i]) == ("episode" in w_info), (t, i)
                if "episode" in w_info:
                    assert (infos[i]["episode"]["r"], infos[i]["episode"]["l"]) == (w_info["episode"]["r"], w_info["episode"]["l"]), (t, i)
                    episodes += 1
            for i in np.flatnonzero(done):
                assert not obs[i, :, :, :9].any() and obs[i, :, :, 9:].any(), (t, i)
                finished += 1
        assert episodes > 0 and finished >= episodes
    finally:
        venv.close()


# ---------------------------------------------------------------------------------------------------------- 8. snapshots
def test_wrapped_rgb_snapshots():
    import torch
    from toybox_b200.wrappers import DeepmindToybox
    n = 6
    env = DeepmindToybox("breakout", n, seeds=21, noop_seed=3, grayscale=False)
    gray = DeepmindToybox("breakout", n, seeds=21, noop_seed=3)
    try:
        env.reset()
        gray.reset()
        for t in range(30):
            env.step(_acts(n, 4, t))
            gray.step(_acts(n, 4, t))
        snap = env.save_state()
        assert tuple(snap.obs.shape) == (n, 4, 84, 84, 3)
        after = []
        for t in range(30, 45):
            env.step(_acts(n, 4, t))
            after.append(env.stacked().cpu().numpy())
        env.load_state(snap)
        for k, t in enumerate(range(30, 45)):
            env.step(_acts(n, 4, t))
            assert np.array_equal(env.stacked().cpu().numpy(), after[k]), t
        env.fork([2])                # env 2 into every env: every ring and state is env 2's
        st = env.stacked().cpu().numpy()
        assert all(np.array_equal(st[i], st[2]) for i in range(n))
        acts = np.full(n, 1, np.int32)
        for t in range(10):
            env.step(acts)
            st = env.stacked().cpu().numpy()
            assert all(np.array_equal(st[i], st[0]) for i in range(n)), t
        # gray into colour and colour into gray: refused before any device work, the envs untouched
        ring, gring = env.obs.clone(), gray.obs.clone()
        with pytest.raises(ValueError, match="of 3 channels .*of 1 channel"):
            env.load_state(gray.save_state())
        with pytest.raises(ValueError, match="of 1 channel .*of 3 channels"):
            gray.load_state(snap)
        assert torch.equal(env.obs, ring) and torch.equal(gray.obs, gring)
        env.check()
        gray.check()
    finally:
        env.close()
        gray.close()
