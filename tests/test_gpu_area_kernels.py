"""GPU tier: every code path of the INTER_AREA (WarpFrame) render -- the direct kernels and the warp-per-env tile
kernel with its list, sweep and per-tile rebuild paths, at up to 5 x 4 and at 8 x 8 taps -- against the oracle's
cv2-exact resize, on mid-game states of all three games and on several output sizes; and the native layouts'
broadcast + patch render with its dense-env hand-over to the canvas kernel."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GAMES = ["breakout", "amidar", "space_invaders"]
TILE = {"TBX_AREA_KERNEL": "tile"}        # Breakout: without the direct kernel (tbx_render_direct.cuh) in front of the tile kernel
VARIANTS = [{}, TILE, dict(TILE, TBX_AREA_DIGIT_CACHE="0"), dict(TILE, TBX_AREA_LCAP="24"), dict(TILE, TBX_AREA_LCAP="3"),
            dict(TILE, TBX_AREA_LCAP="40"), {"TBX_AREA_LCAP": "3"}]
SIZES = [(84, 84), (96, 80), (64, 64), (48, 60), (100, 37)]
# per game: the accepted size with the largest tile-kernel scratch window (8 x 8 taps); each is refused for another game
WORST_SIZE = {"breakout": (32, 20), "space_invaders": (40, 28), "amidar": (23, 35)}


def _advance(tbx, oracle_mod, game, n, steps, seed):
    pool = tbx.BatchedToybox(game, n, seeds=seed)
    ref = oracle_mod.OracleBatch(game, n, seeds=seed + np.arange(n))
    legal = np.asarray(oracle_mod.LEGAL[game], np.int32)
    for t in range(steps):
        acts = legal[[oracle_mod.action_index(0xB200, i, t, len(legal)) for i in range(n)]]
        if game == "breakout":          # track the ball with an aim error so that bricks get broken
            for i in range(n):
                s = ref.states[i]
                if s.is_dead:
                    acts[i] = 1
                elif i % 4:
                    bx = s.balls[0].position.x if s.n_balls else 120.0
                    off = ((i * 7 + t // 50) % 9) - 4
                    acts[i] = 3 if bx + off > s.paddle.position.x + 1 else 4 if bx + off < s.paddle.position.x - 1 else 0
        pool.apply_ale_action(acts, auto_reset=True)
        ref.step(acts, auto_reset=True)
    return pool, ref


def _set_env(v):
    for k in ("TBX_AREA_LCAP", "TBX_AREA_KERNEL", "TBX_AREA_DIGIT_CACHE"):
        os.environ.pop(k, None)
    os.environ.update(v)


@pytest.mark.parametrize("game", GAMES)
def test_area_render_paths_bit_exact(tbx, oracle_mod, game):
    n = 45                                   # ragged: the last chunk holds 5 envs
    pool, ref = _advance(tbx, oracle_mod, game, n, 1200 if game == "breakout" else 400, 77)
    try:
        for ow, oh in SIZES + [WORST_SIZE[game]]:
            want = ref.render("gray84", ow, oh).reshape(n, -1)
            for v in VARIANTS:
                _set_env(v)
                got = pool.render(obs=("gray_area", ow, oh)).cpu().numpy().reshape(n, -1)
                bad = np.argwhere(got != want)
                assert bad.size == 0, (game, ow, oh, v, bad[:5], got[tuple(bad[0])], want[tuple(bad[0])])
    finally:
        _set_env({})
        pool.close()


@pytest.mark.parametrize("game", GAMES)
def test_native_render_paths_bit_exact(tbx, oracle_mod, game):
    """native layouts: broadcast + patch with its dense-env hand-over to the canvas kernel (never / always / mixed; Breakout and
    Amidar -- Space Invaders is always patched)"""
    n = 45
    pool, ref = _advance(tbx, oracle_mod, game, n, 1200 if game == "breakout" else 400, 78)
    try:
        for mode in ("rgb", "rgba", "gray"):
            want = ref.render(mode).reshape(n, -1)
            for v in ({}, {"TBX_NATIVE_DENSE": "-1"}, {"TBX_NATIVE_DENSE": "0"}, {"TBX_NATIVE_DENSE": "3"}):
                os.environ.pop("TBX_NATIVE_DENSE", None)
                os.environ.update(v)
                got = pool.render(obs=mode).cpu().numpy().reshape(n, -1)
                bad = np.argwhere(got != want)
                assert bad.size == 0, (game, mode, v, bad[:5], got[tuple(bad[0])], want[tuple(bad[0])])
    finally:
        os.environ.pop("TBX_NATIVE_DENSE", None)
        pool.close()


@pytest.mark.parametrize("game", GAMES)
def test_hud_digit_patches_every_value(tbx, oracle_mod, game):
    """pre-resolved HUD digit patches: every digit value in every decimal position (isolated single digits use the
    patch, multi-digit numbers fall back to the tiles), on fresh and on advanced games, several output sizes"""
    n = 64
    pool, ref = _advance(tbx, oracle_mod, game, n, 120, 90)
    scores = [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 19, 70, 100, 305, 999, 1000, 4821, 90909, 123456, 7654321, 10 ** 9] * 3
    scores = np.asarray(scores[:n], np.int64)
    lives = 1 + (np.arange(n) % 9)
    try:
        pool.set_property("score", scores.astype(np.int32))
        pool.set_property("lives", lives.astype(np.int32))
        if game == "amidar":
            pool.set_property("jumps", (np.arange(n) % 10).astype(np.int32))
        if game == "space_invaders":
            pool.set_property("life_display_timer", (np.arange(n) % 2) * 30)
        for i in range(n):
            js = ref.state_json(i)
            js["score"] = int(scores[i]); js["lives"] = int(lives[i])
            if game == "amidar":
                js["jumps"] = int(i % 10)
            if game == "space_invaders":
                js["life_display_timer"] = int((i % 2) * 30)
            ref.write_state_json(i, js)
        for ow, oh in ((84, 84), (96, 80), (64, 64)):
            want = ref.render("gray84", ow, oh).reshape(n, -1)
            for v in ({}, TILE, dict(TILE, TBX_AREA_DIGIT_CACHE="0")):
                _set_env(v)
                got = pool.render(obs=("gray_area", ow, oh)).cpu().numpy().reshape(n, -1)
                bad = np.argwhere(got != want)
                assert bad.size == 0, (game, ow, oh, v, bad[:5], got[tuple(bad[0])], want[tuple(bad[0])])
    finally:
        _set_env({})
        pool.close()


def test_direct_kernel_mixed_pool(tbx, oracle_mod):
    """Breakout's direct INTER_AREA kernel on a pool that mixes the states it covers (worn walls, several balls, wide and
    misplaced paddles, multi-digit scores) with states it hands to the tile kernel (custom brick tables, a ball inside the
    HUD rows, scores whose digits are clipped by the frame) -- every env must come out bit-exact, twice in a row (the
    hand-over list empties itself), and again after further steps."""
    n = 203
    pool, ref = _advance(tbx, oracle_mod, "breakout", n, 300, 5)
    rng = np.random.default_rng(11)
    states = []
    for i in range(n):
        js = ref.state_json(i)
        for k in rng.choice(108, size=int(rng.integers(0, 108)) if i % 3 else 0, replace=False):
            js["bricks"][int(k)]["alive"] = False
        if i % 5 == 1:
            js["balls"] = [{"position": {"x": float(rng.uniform(0, 240)), "y": float(rng.uniform(20, 170))}, "velocity": {"x": 1.0, "y": -1.0}}
                           for _ in range(int(rng.integers(0, 5)))]
        if i % 7 == 2:
            js["paddle"]["position"] = {"x": float(rng.uniform(0, 240)), "y": float(rng.choice([143.0, 60.0, 50.5, 158.0]))}
            js["paddle_width"] = float(rng.choice([24.0, 48.0, 7.0, 300.0]))
            js["ball_radius"] = float(rng.choice([2.0, 5.5, 0.5]))
        js["score"] = int(rng.choice([0, 7, 42, 860, 123456, 123456789]))
        js["lives"] = int(rng.choice([5, 1, 13]))
        if i % 11 == 3:
            js["bricks"][int(rng.integers(108))]["position"]["x"] += 3.0          # a custom brick table: the tile kernel's env
        if i % 13 == 4:
            js["balls"] = [{"position": {"x": 100.0, "y": 5.0}, "velocity": {"x": 1.0, "y": 1.0}}]   # inside the HUD rows
        ref.write_state_json(i, js)
        states.append(js)
    pool.write_state_json(states)
    legal = np.asarray(oracle_mod.LEGAL["breakout"], np.int32)
    try:
        for rnd in range(3):
            for ow, oh in ((84, 84), (96, 80), (64, 64)):
                want = ref.render("gray84", ow, oh).reshape(n, -1)
                for v in ({}, {}, TILE):
                    _set_env(v)
                    got = pool.render(obs=("gray_area", ow, oh)).cpu().numpy().reshape(n, -1)
                    bad = np.argwhere(got != want)
                    assert bad.size == 0, (rnd, ow, oh, v, bad[:5], got[tuple(bad[0])], want[tuple(bad[0])])
            for t in range(40):
                acts = legal[[oracle_mod.action_index(0xB200, i, 1000 * rnd + t, len(legal)) for i in range(n)]]
                pool.apply_ale_action(acts, auto_reset=True)
                ref.step(acts, auto_reset=True)
    finally:
        _set_env({})
        pool.close()


def test_si_direct_kernel_adversarial_states(tbx, oracle_mod):
    """Space Invaders' direct INTER_AREA kernel (sparse sprites: patches for isolated bank sprites, pixel-by-pixel evaluation
    for the rest) on states built to hit every branch: sprites clipped by the frame, invaders moved on top of each other / of
    shields / of lasers, eroded shields, non-default colours (no patch set), the ufo, explosions, huge lasers, lives display,
    multi-digit scores, shields and ship pushed into the ground line -- bit-exact against the oracle, several output sizes."""
    n = 96
    pool, ref = _advance(tbx, oracle_mod, "space_invaders", n, 300, 21)
    rng = np.random.default_rng(4)
    states = []
    for i in range(n):
        js = ref.state_json(i)
        k = i % 12
        if k == 1:
            for e in js["enemies"][:8]:
                e["x"], e["y"] = int(rng.integers(-12, 316)), int(rng.integers(-8, 205))
        elif k == 2:
            for e in js["enemies"][6:18]:
                e["x"], e["y"] = js["shields"][0]["x"] + int(rng.integers(-10, 10)), js["shields"][0]["y"] + int(rng.integers(-8, 12))
        elif k == 3:
            js["enemy_lasers"] = [{"x": int(rng.integers(0, 318)), "y": int(rng.integers(0, 190)), "w": 2, "h": 8, "t": 0, "movement": "Down", "speed": 3,
                                   "color": {"r": 252, "g": 252, "b": 84, "a": 255}} for _ in range(4)]
            js["ship_laser"] = {"x": js["enemies"][7]["x"] + 3, "y": js["enemies"][7]["y"] + 2, "w": 2, "h": 8, "t": 0, "movement": "Up", "speed": 8,
                                "color": {"r": 35, "g": 129, "b": 59, "a": 255}}
        elif k == 4:
            js["ufo"]["appearance_counter"] = None
            js["ufo"]["x"] = int(rng.integers(-2, 318))
            js["ship"]["color"] = {"r": 200, "g": 10, "b": 90, "a": 255}
        elif k == 5:
            js["enemy_lasers"] = [{"x": 20, "y": 10, "w": 280, "h": 150, "t": 0, "movement": "Down", "speed": 3, "color": {"r": 9, "g": 99, "b": 199, "a": 255}}]
        elif k == 6:
            js["life_display_timer"] = 40
            js["lives"] = int(rng.choice([3, 27, 104]))
            js["score"] = int(rng.choice([0, 35, 1250, 99999, 1234567]))
        elif k == 7:
            for sh in js["shields"]:
                for row in sh["data"]:
                    for c in rng.choice(16, size=6, replace=False):
                        row[int(c)] = {"r": 0, "g": 0, "b": 0, "a": 0}
            js["shields"][1]["x"], js["shields"][1]["y"] = int(rng.integers(-8, 310)), int(rng.integers(170, 200))
        elif k == 8:
            js["ship"]["x"], js["ship"]["y"] = int(rng.integers(-10, 315)), int(rng.integers(180, 206))
            for e in js["enemies"][:6]:
                e["alive"] = False
                e["death_counter"] = 5
        elif k == 9:
            js["ufo"]["appearance_counter"] = None
            js["ufo"]["death_counter"] = 9
            js["ship"]["alive"] = False
            js["ship"]["death_counter"] = 12
        elif k == 10:
            for j, e in enumerate(js["enemies"]):
                e["x"], e["y"] = 40 + 17 * (j % 12), 30 + 11 * (j // 12)          # packed: neighbours share output pixels
        ref.write_state_json(i, js)
        states.append(js)
    pool.write_state_json(states)
    legal = np.asarray(oracle_mod.LEGAL["space_invaders"], np.int32)
    try:
        for rnd in range(2):
            for ow, oh in ((84, 84), (96, 80), (64, 64), (48, 60)):
                want = ref.render("gray84", ow, oh).reshape(n, -1)
                for v in ({}, TILE):
                    _set_env(v)
                    got = pool.render(obs=("gray_area", ow, oh)).cpu().numpy().reshape(n, -1)
                    bad = np.argwhere(got != want)
                    assert bad.size == 0, (rnd, ow, oh, v, bad[:5], got[tuple(bad[0])], want[tuple(bad[0])])
            for mode in ("rgb", "gray", "rgba"):              # native layouts: broadcast + patch
                want = ref.render(mode).reshape(n, -1)
                got = pool.render(obs=mode).cpu().numpy().reshape(n, -1)
                bad = np.argwhere(got != want)
                assert bad.size == 0, (rnd, mode, bad[:5], got[tuple(bad[0])], want[tuple(bad[0])])
            for t in range(30):
                acts = legal[[oracle_mod.action_index(0xB200, i, 500 + t, len(legal)) for i in range(n)]]
                pool.apply_ale_action(acts, auto_reset=True)
                ref.step(acts, auto_reset=True)
    finally:
        _set_env({})
        pool.close()


def test_amidar_painted_corridors_every_layout(tbx, oracle_mod):
    """late-game Amidar boards (long painted corridors, painted boxes, moved / removed / caught enemies, off-board player): the
    direct kernel's tile-look grid and the tile kernel's merged runs; every layout and renderer against the oracle"""
    n = 24
    pool, ref = _advance(tbx, oracle_mod, "amidar", n, 60, 12)
    rng = np.random.default_rng(5)
    states = []
    for i in range(n):
        js = ref.state_json(i)
        tiles = js["board"]["tiles"]
        for _ in range(2 + i):                                   # paint random horizontal / vertical stretches of track
            ty, tx, ln, horiz = int(rng.integers(31)), int(rng.integers(32)), int(rng.integers(1, 20)), bool(rng.integers(2))
            for k in range(ln):
                y, x = (ty, tx + k) if horiz else (ty + k, tx)
                if y < 31 and x < 32 and tiles[y][x] in ("Unpainted", "ChaseMarker"):
                    tiles[y][x] = "Painted"
        for b in js["board"]["boxes"][: i % 7]:
            b["painted"] = True
        if i % 5 == 1:
            js["player"]["position"] = {"x": int(rng.integers(-200, 2200)), "y": int(rng.integers(-200, 2600))}
            for e in js["enemies"][:3]:
                e["position"] = {"x": int(rng.integers(0, 1984)), "y": int(rng.integers(0, 2400))}
        if i % 5 == 2:
            js["enemies"] = js["enemies"][:2]
            js["enemies"][0]["caught"] = True
            js["score"], js["lives"], js["jumps"] = int(rng.integers(0, 99999)), int(rng.integers(0, 20)), int(rng.integers(0, 10))
        if i % 5 == 3:
            for row in tiles[::3]:
                for x in range(0, 32, 2):
                    row[x] = "Empty" if row[x] != "Empty" else "Unpainted"           # checkerboard damage: every look next to every other
        ref.write_state_json(i, js)
        states.append(js)
    pool.write_state_json(states)
    keys = ("TBX_NATIVE_DENSE", "TBX_AREA_LCAP", "TBX_AREA_KERNEL")
    try:
        for mode, omode in (("gray84", "gray84"), ("rgb", "rgb"), ("gray", "gray"), ("rgba", "rgba")):
            want = ref.render(omode).reshape(n, -1)
            for v in ({}, TILE, {"TBX_NATIVE_DENSE": "0"}, {"TBX_NATIVE_DENSE": "-1"}, {"TBX_NATIVE_DENSE": "4"}, dict(TILE, TBX_AREA_LCAP="16")):
                for k in keys:
                    os.environ.pop(k, None)
                os.environ.update(v)
                got = pool.render(obs=mode).cpu().numpy().reshape(n, -1)
                bad = np.argwhere(got != want)
                assert bad.size == 0, (mode, v, bad[:5], got[tuple(bad[0])], want[tuple(bad[0])])
    finally:
        for k in keys:
            os.environ.pop(k, None)
        pool.close()


def test_si_score_strip_every_digit_pair(tbx, oracle_mod):
    """Space Invaders' score is rendered as one strip from a table of digit pairs (neighbouring digits feed a common output column):
    scores that put every pair of digits (and the empty slot) next to each other at every position, ten-digit scores, and states where
    something else reaches into the strip (a laser, an invader: the digits are then evaluated with it) -- bit-exact, several sizes."""
    scores = [0, 7, 10, 99, 100, 101, 909, 1000, 4711, 10000, 99999, 100000, 1234567, 7654321, 10000000, 98765432, 100000000, 123456789,
              999999999, 1000000000, 1999999999, 2000000000, 2147483647]
    for k in range(9):                     # digit a in slot k, digit b in slot k + 1, a leading 1 above where b is 0
        for a in range(10):
            for b in range(10):
                v = a * 10 ** k + b * 10 ** (k + 1) + (10 ** (k + 2) if b == 0 and k + 2 <= 9 else 0)
                if 0 < v <= 2147483647:
                    scores.append(v)
    scores = sorted(set(scores))
    n = len(scores)
    pool, ref = _advance(tbx, oracle_mod, "space_invaders", n, 40, 77)
    rng = np.random.default_rng(9)
    states = []
    for i in range(n):
        js = ref.state_json(i)
        js["score"] = int(scores[i])
        if i % 9 == 4:        # a laser through the score's rows
            js["enemy_lasers"] = [{"x": int(rng.integers(40, 122)), "y": int(rng.integers(0, 8)), "w": 2, "h": 8, "t": 0, "movement": "Down", "speed": 3,
                                   "color": {"r": 252, "g": 252, "b": 84, "a": 255}}]
        if i % 9 == 7:        # an invader on top of it
            js["enemies"][3]["x"], js["enemies"][3]["y"] = int(rng.integers(30, 120)), int(rng.integers(0, 6))
        ref.write_state_json(i, js)
        states.append(js)
    pool.write_state_json(states)
    try:
        for ow, oh in ((84, 84), (96, 80), (64, 64), (48, 60), (128, 128)):
            want = ref.render("gray84", ow, oh).reshape(n, -1)
            for v in ({}, TILE):
                _set_env(v)
                got = pool.render(obs=("gray_area", ow, oh)).cpu().numpy().reshape(n, -1)
                bad = np.argwhere(got != want)
                assert bad.size == 0, (ow, oh, v, [scores[int(b[0])] for b in bad[:5]], bad[:5], got[tuple(bad[0])], want[tuple(bad[0])])
    finally:
        _set_env({})
        pool.close()
