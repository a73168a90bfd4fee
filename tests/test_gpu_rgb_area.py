"""GPU tier: the colour INTER_AREA layout (TBX_OBS_RGB_AREA, obs 'rgb84' / ('rgb_area', w, h)), rendered by the tile kernel's
RGB mode, bit for bit against the oracle's cv2-exact 3-channel resize of its RGB frame (test_rgb_area_cpu.rgb_area).  Every render goes into a buffer filled with 0xA5
first, so that a pixel the kernel skips cannot pass on a previous render's bytes.

Covered: the list, sweep and per-tile rebuild paths at every tap count (3..5 x 3..4 and 8 x 8); colours that differ in RGB but
share a gray (any use of the luma or of a gray-keyed table in the RGB path shows there); RGB renders interleaved with the gray
direct kernel and its hand-over to the tile kernel; a pool of many CTAs; tbx_step_host, BatchedToyboxEnv and CUDA-graph
capture; and the sizes the layout refuses, which are exactly the gray layout's."""
import os

import numpy as np
import pytest

from test_gpu_area_coverage import _advance_cfg, _assert_same, _breakout_mixed, _brk_cfg, _col, _render_check, _si_adversarial
from test_gpu_area_kernels import _advance
from test_rgb_area_cpu import rgb_area

pytestmark = pytest.mark.gpu
GAMES = ["breakout", "amidar", "space_invaders"]
KEYS = ("TBX_AREA_LCAP", "TBX_AREA_KERNEL", "TBX_AREA_DIGIT_CACHE", "TBX_DIRECT_GRID")
SIZES = [(84, 84), (64, 64), (96, 80), (92, 83), (128, 128), (100, 37)]
# per game: the accepted size with the largest tile-kernel scratch window (8 x 8 taps)
WORST_SIZE = {"breakout": (32, 20), "space_invaders": (40, 28), "amidar": (23, 35)}
# default list, two capacities that force the sweeps, and 3, which also forces the per-tile rebuild
LCAPS = [{}, {"TBX_AREA_LCAP": "24"}, {"TBX_AREA_LCAP": "40"}, {"TBX_AREA_LCAP": "3"}]


def _set(v):
    for k in KEYS:
        os.environ.pop(k, None)
    os.environ.update(v)


def _rgb_check(pool, ref, n, size, what):
    import torch
    ow, oh = size
    want = rgb_area(ref_oracle(), ref.render("rgb"), ow, oh).reshape(n, oh, ow * 3)
    out = torch.full((n, oh, ow, 3), 0xA5, dtype=torch.uint8, device=pool.device)
    got = pool.render(out=out, obs=("rgb_area", ow, oh)).cpu().numpy().reshape(n, oh, ow * 3)
    _assert_same(got, want, "%s rgb %dx%d (x = 3 * pixel + channel)" % (what, ow, oh))


def ref_oracle():
    from oracle import oracle
    return oracle


def _luma(c):
    return int(0.299 * c[0] + 0.587 * c[1] + 0.114 * c[2])


def _twin(c):
    """a colour far from `c` in RGB with the same gray byte"""
    for db in (90, -90, 60, -60):
        for dg in range(-30, 31):
            for dr in range(-6, 7):
                t = (c[0] + dr, c[1] + dg, c[2] + db)
                if all(0 <= v <= 255 for v in t) and _luma(t) == _luma(c):
                    return t
    raise AssertionError(c)


# ----------------------------------------------------------------------------------------------------------- 1. paths
@pytest.mark.parametrize("game", GAMES)
def test_rgb_area_paths_bit_exact(tbx, oracle_mod, game):
    n = 45                                   # ragged: the last CTA holds 5 envs
    pool, ref = _advance(tbx, oracle_mod, game, n, 800 if game == "breakout" else 300, 77)
    try:
        for size in SIZES + [WORST_SIZE[game]]:
            for v in LCAPS:
                _set(v)
                _rgb_check(pool, ref, n, size, "%s %s" % (game, v or "default"))
        pool.check()
    finally:
        _set({})
        pool.close()


# ---------------------------------------------------------------------------------------- 2. colours that share a gray
def _brk_twin_cfg():
    """brick rows in pairs of one gray (the second row of a pair: the twin of the first), one row of gray 0 on the black
    background, and paddle and ball in two colours of one gray"""
    a, b = (200, 72, 72), (66, 72, 200)
    rows = [a, _twin(a), b, _twin(b), (0, 0, 1), (72, 160, 72)]
    p = (30, 200, 250)
    return _brk_cfg(row_colors=[_col(*c) for c in rows], paddle_color=_col(*p), ball_color=_col(*_twin(p)))


def _ami_twin_cfg():
    """painted track in a colour of the unpainted track's gray, enemies in a third colour of that gray"""
    import emu_lib
    cfg = emu_lib.Emu("amidar").config_json()
    u = cfg["unpainted_color"]
    painted = _twin((u["r"], u["g"], u["b"]))
    cfg.update(painted_color=_col(*painted), enemy_color=_col(*_twin(painted)))
    return cfg


@pytest.mark.parametrize("case", ["breakout_rows_paddle_ball", "breakout_custom_tables", "amidar", "space_invaders"])
def test_rgb_area_colours_sharing_a_gray(tbx, oracle_mod, case):
    """configs whose colours are distinct in RGB and equal in gray; Breakout also with a custom brick table in every env (no env
    on base frame 1); Space Invaders on the gray tests' adversarial states (sprites clipped, stacked, recoloured)"""
    n = 24
    rng = np.random.default_rng(3)
    if case.startswith("breakout"):
        cfg = _brk_twin_cfg()
        assert _luma((0, 0, 1)) == 0
        pool, ref = _advance_cfg(tbx, oracle_mod, "breakout", cfg, n, 300, 41)
        states = []
        for i in range(n):
            js = ref.state_json(i)
            for k in rng.choice(len(js["bricks"]), size=int(rng.integers(0, 60)), replace=False):
                js["bricks"][int(k)]["alive"] = False
            if case == "breakout_custom_tables":
                js["bricks"][i % len(js["bricks"])]["position"]["x"] += 2.0
            if i % 3 == 1:               # the ball over the paddle: the two colours of one gray side by side
                js["balls"] = [{"position": {"x": js["paddle"]["position"]["x"], "y": 140.0}, "velocity": {"x": 1.0, "y": 1.0}}]
            ref.write_state_json(i, js)
            states.append(js)
        pool.write_state_json(states)
        game = "breakout"
    elif case == "amidar":
        pool, ref = _advance_cfg(tbx, oracle_mod, "amidar", _ami_twin_cfg(), n, 200, 42)
        states = []
        for i in range(n):
            js = ref.state_json(i)
            tiles = js["board"]["tiles"]
            for _ in range(4 + i):
                ty, tx, ln = int(rng.integers(31)), int(rng.integers(32)), int(rng.integers(1, 20))
                for k in range(ln):
                    if tx + k < 32 and tiles[ty][tx + k] in ("Unpainted", "ChaseMarker"):
                        tiles[ty][tx + k] = "Painted"
            ref.write_state_json(i, js)
            states.append(js)
        pool.write_state_json(states)
        game = "amidar"
    else:
        pool, ref = _si_adversarial(tbx, oracle_mod, n, 23)
        game = "space_invaders"
    try:
        for rnd in range(2):
            for size in ((84, 84), (64, 64), (96, 80), WORST_SIZE[game]):
                for v in ({}, {"TBX_AREA_LCAP": "3"}):
                    _set(v)
                    _rgb_check(pool, ref, n, size, "%s round %d %s" % (case, rnd, v or "default"))
            _set({})
            legal = np.asarray(oracle_mod.LEGAL[game], np.int32)
            for t in range(20):
                acts = legal[[oracle_mod.action_index(0xB200, i, 900 + t, len(legal)) for i in range(n)]]
                pool.apply_ale_action(acts, auto_reset=True)
                ref.step(acts, auto_reset=True)
        pool.check()
    finally:
        _set({})
        pool.close()


# ------------------------------------------------------------------------------------------------------- 3. interleaving
def test_rgb_area_interleaved_with_gray_direct_kernel(tbx, oracle_mod):
    """a Breakout pool that mixes envs the gray direct kernel covers with envs it hands over (custom brick tables, a ball in the
    HUD rows): gray84, rgb84, rgb 64x64, gray84 again, a few steps, and again -- the RGB renders must leave the hand-over
    counters and the per-size caches as the gray renders expect them"""
    n = 67
    pool, ref = _breakout_mixed(tbx, oracle_mod, n, 8)
    legal = np.asarray(oracle_mod.LEGAL["breakout"], np.int32)
    try:
        for rnd in range(3):
            _render_check(pool, ref, n, (84, 84), "round %d gray first" % rnd)
            _rgb_check(pool, ref, n, (84, 84), "round %d" % rnd)
            _rgb_check(pool, ref, n, (64, 64), "round %d" % rnd)
            _render_check(pool, ref, n, (84, 84), "round %d gray after rgb" % rnd)
            for t in range(15):
                acts = legal[[oracle_mod.action_index(0xB200, i, 300 * rnd + t, len(legal)) for i in range(n)]]
                pool.apply_ale_action(acts, auto_reset=True)
                ref.step(acts, auto_reset=True)
        pool.check()
    finally:
        pool.close()


# ------------------------------------------------------------------------------------------------------- 4. many CTAs
def test_rgb_area_many_ctas(tbx, oracle_mod):
    import torch
    n = 3000
    pool = tbx.BatchedToybox("breakout", n, seeds=5)
    ref = oracle_mod.OracleBatch("breakout", n, seeds=5 + np.arange(n))
    acts = torch.empty(n, dtype=torch.int32, device=pool.device)
    try:
        for t in range(120):
            pool.fill_random_actions(acts, 0xB200, t)
            pool.apply_ale_action(acts, auto_reset=True)
            ref.step(acts.cpu().numpy(), auto_reset=True)
        _rgb_check(pool, ref, n, (84, 84), "3000 envs")
        pool.check()
    finally:
        pool.close()


# -------------------------------------------------------------------------------------------------- 5. other entry points
def test_rgb_area_step_host_and_env(tbx, oracle_mod):
    """tbx_step_host with rgb84 = step + render; BatchedToyboxEnv(obs='rgb84') reports (84, 84, 3) and steps to the oracle's frames"""
    import torch
    from toybox_b200.envs.atari import BatchedToyboxEnv
    n = 16
    a = tbx.BatchedToybox("amidar", n, obs="rgb84", seeds=3)
    b = tbx.BatchedToybox("amidar", n, obs="rgb84", seeds=3)
    ref = oracle_mod.OracleBatch("amidar", n, seeds=3 + np.arange(n))
    legal = np.asarray(oracle_mod.LEGAL["amidar"], np.int32)
    try:
        assert a.obs_shape == (84, 84, 3)
        for t in range(60):
            acts = legal[[oracle_mod.action_index(0xB200, i, t, len(legal)) for i in range(n)]]
            obs_h, r, d, _ = a.step_host(acts)
            obs_d, _, _, _ = b.step(torch.as_tensor(acts))
            ref.step(acts, auto_reset=True)
            assert obs_h.shape == (n, 84, 84, 3) and np.array_equal(obs_h.numpy(), obs_d.cpu().numpy()), t
            if t % 20 == 19:
                assert np.array_equal(obs_h.numpy(), rgb_area(ref_oracle(), ref.render("rgb"), 84, 84)), t
    finally:
        a.close()
        b.close()
    env = BatchedToyboxEnv("space_invaders", 8, obs="rgb84", seed=1)
    try:
        assert env.toybox.obs_shape == (84, 84, 3) and tuple(env.observation_space.shape) == (84, 84, 3)
        obs = env.reset()
        assert tuple(obs.shape) == (8, 84, 84, 3)
        obs, _, _, _ = env.step(torch.zeros(8, dtype=torch.int64, device=env.device))
        assert tuple(obs.shape) == (8, 84, 84, 3)
    finally:
        env.close()


def test_rgb_area_cuda_graph_replay(tbx):
    """after one warm-up render, step_random + RGB render captured in a CUDA graph replays bit-identically to eager calls"""
    import torch
    n = 64
    g_pool = tbx.BatchedToybox("space_invaders", n, seeds=12)
    e_pool = tbx.BatchedToybox("space_invaders", n, seeds=12)
    out = torch.empty((n, 84, 84, 3), dtype=torch.uint8, device=g_pool.device)
    try:
        g_pool.render(out=out, obs="rgb84")
        torch.cuda.synchronize()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(s):
            with torch.cuda.graph(graph, stream=s):
                g_pool.step_random(99, 5)
                g_pool.render(out=out, obs="rgb84")
        torch.cuda.current_stream().wait_stream(s)
        e_pool.render(obs="rgb84")
        for k in range(12):
            graph.replay()
            e_pool.step_random(99, 5)
            want = e_pool.render(obs="rgb84")
            torch.cuda.synchronize()
            assert torch.equal(out, want), k
    finally:
        g_pool.close()
        e_pool.close()


# ---------------------------------------------------------------------------------------------------------- 6. refusals
def _outcome(pool, mode, size):
    """"ok", or the refusal's message with the layout's name taken out"""
    try:
        pool.render(obs=(mode, size[0], size[1]))
        return "ok"
    except Exception as e:
        return str(e).replace(mode, "<layout>")


@pytest.mark.parametrize("game", GAMES)
def test_rgb_area_refuses_what_gray_refuses(tbx, game):
    """Breakout 120 x 80 (OpenCV's integer-scale fast path), a 129-wide size, and a sweep of sizes: the RGB layout accepts a
    size exactly when the gray layout does, and refuses it with the same message"""
    pool = tbx.BatchedToybox(game, 2, seeds=1)
    try:
        if game == "breakout":
            for size in ((120, 80), (129, 84)):
                gray, rgb = _outcome(pool, "gray_area", size), _outcome(pool, "rgb_area", size)
                assert gray != "ok" and rgb == gray, (size, gray, rgb)
        n_ok = 0
        for w in (8, 23, 40, 64, 84, 100, 128, 129):
            for h in (20, 35, 37, 80, 105, 128):
                gray, rgb = _outcome(pool, "gray_area", (w, h)), _outcome(pool, "rgb_area", (w, h))
                assert gray == rgb, (game, w, h, gray, rgb)
                n_ok += gray == "ok"
        assert 0 < n_ok < 48, n_ok
    finally:
        pool.close()
