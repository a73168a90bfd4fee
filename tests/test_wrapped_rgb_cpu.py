"""CPU tier: the reference for colour observations of the fused wrapper stack (DeepmindToybox(grayscale=False), tbx_wrap_step
under TBX_OBS_RGB_AREA) -- WarpFrame(grayscale=False) (baselines atari_wrappers.py:230-244) in the oracle-side wrapper chain:

  ColourWrappedEnv = oracle.wrappers.WrappedEnv with the base env returning the oracle's RGB frame (ToyboxBaseEnv with
  grayscale=False, envs/atari/base.py:109), MaxAndSkipEnv buffering (H, W, 3) frames, and WarpFrame's resize taken with 3
  interleaved channels (oracle/common.c:tbo_resize_area_u8, cn = 3, = cv2's 3-channel INTER_AREA; test_rgb_area_cpu pins it
  to cv2).  Everything else -- no-op resets, frame skip, EpisodicLife, FireReset, ClipReward, FrameStack, Monitor -- is the
  gray chain's code unchanged, so the gray reference stays exactly what it is.

Checked here: the chain's newest observation is cv2.resize(np.maximum(A, B), (w, h), INTER_AREA) of its last two RGB frames
A and B (max first, then resize: INTER_AREA does not commute with the max); its rewards, dones, lives and scores are the gray
chain's; and DeepmindToybox.stacked()'s colour layout is np.concatenate(frames, axis=-1) of the ring in FrameStack order.
tests/test_gpu_wrapped_rgb.py compares the GPU with ColourWrappedEnv."""
import numpy as np
import pytest

from test_rgb_area_cpu import rgb_area


def colour_wrapped_env(game, seed, config=None, **kw):
    """oracle.wrappers.WrappedEnv(game, seed, **kw) with WarpFrame(grayscale=False): step() / reset() return the frames oldest
    first as uint8[k, h, w, 3].  config: a game config (JSON dict) for the env underneath."""
    from oracle import oracle as O
    from oracle import wrappers as OW

    class ColourWrappedEnv(OW.WrappedEnv):
        def _warp(self, obs):
            return rgb_area(O, obs, self.size[0], self.size[1])

    env = ColourWrappedEnv(game, seed, **kw)
    base = env.base
    if config is not None:                                     # nothing has run yet: swap in the configured engine
        base.b = O.OracleBatch(game, 1, seeds=np.asarray([seed], np.uint32), cfg_json=config)
    base._obs = lambda: base.b.render("rgb")[0]                 # ToyboxBaseEnv(grayscale=False): the RGB frame
    env.skipper._obs_buffer = np.zeros(env.skipper._obs_buffer.shape + (3,), np.uint8)
    return env


def _cv2():
    try:
        import cv2
        return cv2
    except ImportError:
        return None


@pytest.mark.parametrize("game,kw", [("breakout", {}), ("amidar", {}), ("space_invaders", {}),
                                     ("breakout", dict(frame_skip=2, size=(64, 72), frame_stack=3, stack_reset="zero")),
                                     ("space_invaders", dict(frame_skip=1, noop_max=0, size=(64, 64)))])
def test_colour_chain_is_the_resize_of_the_max_of_two_rgb_frames(oracle_mod, game, kw):
    from oracle import wrappers as OW
    cv2 = _cv2()
    w, h = kw.get("size", (84, 84))
    skip = kw.get("frame_skip", 4)
    col = colour_wrapped_env(game, 31, env_id=2, noop_seed=5, **kw)
    gray = OW.WrappedEnv(game, 31, env_id=2, noop_seed=5, **kw)
    ob = col.reset()
    assert ob.shape == (kw.get("frame_stack", 4), h, w, 3) and ob.dtype == np.uint8
    gray.reset()
    n_act = len(col.base.legal)
    checked = 0
    for t in range(120 if game == "breakout" else 60):
        a = oracle_mod.action_index(0xB200, 2, t, n_act)
        c_obs, c_rew, c_done, c_info = col.step(a)
        g_obs, g_rew, g_done, g_info = gray.step(a)
        assert (c_rew, c_done, c_info["lives"], c_info["score"]) == (g_rew, g_done, g_info["lives"], g_info["score"]), t
        if c_done or not c_info["fresh"]:
            continue
        A, B = col.skipper._obs_buffer
        if skip == 1:
            assert np.array_equal(A, B)
        want = rgb_area(oracle_mod, np.maximum(A, B), w, h)
        assert np.array_equal(c_obs[-1], want), t
        if cv2 is not None:
            assert np.array_equal(c_obs[-1], cv2.resize(np.maximum(A, B), (w, h), interpolation=cv2.INTER_AREA)), t
        checked += 1
    assert checked > 10


def _ring_env(n, k, h, w, grayscale, slot):
    """a DeepmindToybox shell on the CPU with a given ring: stacked() is plain tensor work"""
    import torch
    from toybox_b200.wrappers import DeepmindToybox
    env = DeepmindToybox.__new__(DeepmindToybox)
    env.n_envs, env.k, env.out_h, env.out_w, env.grayscale, env.slot, env.device = n, k, h, w, grayscale, slot, torch.device("cpu")
    shape = (n, k, h, w) if grayscale else (n, k, h, w, 3)
    env.obs = torch.as_tensor(np.random.default_rng(k * 10 + slot).integers(0, 256, size=shape, dtype=np.uint8))
    return env


@pytest.mark.parametrize("k,slot", [(4, 0), (4, 2), (3, 1), (1, 0)])
def test_stacked_colour_layout_is_frame_major(k, slot):
    """stacked() in colour = np.concatenate(frames oldest first, axis=-1): [N, h, w, 3k], the oldest frame's R, G, B first (what
    LazyFrames / VecFrameStack give for (h, w, 3) frames); in gray it is unchanged, np.stack(frames, axis=-1)"""
    n, h, w = 3, 7, 5
    env = _ring_env(n, k, h, w, False, slot)
    ring = env.obs.numpy()
    frames = [ring[:, (slot + 1 + i) % k] for i in range(k)]
    got = env.stacked().numpy()
    assert got.shape == (n, h, w, 3 * k)
    assert np.array_equal(got, np.concatenate(frames, axis=-1))
    assert np.array_equal(got[..., :3], ring[:, (slot + 1) % k]) and np.array_equal(got[..., -3:], ring[:, slot])
    g = _ring_env(n, k, h, w, True, slot)
    gring = g.obs.numpy()
    assert np.array_equal(g.stacked().numpy(), np.stack([gring[:, (slot + 1 + i) % k] for i in range(k)], axis=-1))
