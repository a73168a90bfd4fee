"""GPU tier: the parts of the INTER_AREA (WarpFrame) render that the other render tests do not reach, bit-exact against the
oracle's cv2-exact resize, every env compared:

A. the direct kernels' persistent schedule past its first chunk: small grids (TBX_DIRECT_GRID) make every team draw further
   chunks from the device-wide counter, fill the hand-over list across chunks, and re-arm the counter for the next launch;
B. a hand-over list longer than the env-list tile kernel's grid (296 CTAs x 8 envs), so that its loop takes a second pass;
C. edited configs through the direct kernels (brick-row counts up to the 144-brick capacity, colours, an edited Amidar
   board, moved Space Invaders shields, sizes with and without sprite patch tables), with the direct coverage of every
   (config, size) confirmed through the builders themselves (emu_lib.Emu.direct_info);
D. the wrapped path's dual tile kernel (max of two frames) under list overflow, without digit patches, on intervened states.

The test-only switches (TBX_DIRECT_GRID, TBX_AREA_LCAP, TBX_AREA_KERNEL, TBX_AREA_DIGIT_CACHE) are read at every render."""
import copy
import os

import numpy as np
import pytest

import emu_lib
from test_gpu_area_kernels import TILE, _advance

pytestmark = pytest.mark.gpu
KEYS = ("TBX_AREA_LCAP", "TBX_AREA_KERNEL", "TBX_AREA_DIGIT_CACHE", "TBX_DIRECT_GRID")


def _set(v):
    for k in KEYS:
        os.environ.pop(k, None)
    os.environ.update(v)


def _assert_same(got, want, what):
    """got / want: [n, h, w]; names the failing envs, the first bad pixel and the variant"""
    bad = np.argwhere(got != want)
    if bad.size:
        envs = np.unique(bad[:, 0])
        e, y, x = (int(v) for v in bad[0])
        raise AssertionError("%s: %d env(s) differ, first %s; env %d pixel (y %d, x %d): got %d, want %d"
                             % (what, len(envs), envs[:12].tolist(), e, y, x, got[e, y, x], want[e, y, x]))


def _render_check(pool, ref, n, size, what):
    """renders into a buffer filled with 0xA5 first, so that an env the kernels skip cannot pass on a previous render's bytes"""
    import torch
    ow, oh = size
    want = ref.render("gray84", ow, oh).reshape(n, oh, ow)
    out = torch.full((n, oh, ow), 0xA5, dtype=torch.uint8, device=pool.device)
    got = pool.render(out=out, obs=("gray_area", ow, oh)).cpu().numpy().reshape(n, oh, ow)
    _assert_same(got, want, "%s %dx%d" % (what, ow, oh))


def _covered(game, size, cfg=None):
    info = emu_lib.Emu(game, cfg).direct_info(*size)
    assert info["ok"] == 1, (game, size, info)
    return info


def _step(pool, ref, oracle_mod, game, n, steps, t0):
    legal = np.asarray(oracle_mod.LEGAL[game], np.int32)
    for t in range(steps):
        acts = legal[[oracle_mod.action_index(0xB200, i, t0 + t, len(legal)) for i in range(n)]]
        pool.apply_ale_action(acts, auto_reset=True)
        ref.step(acts, auto_reset=True)


# ---------------------------------------------------------------------------------------------------------------- pools
def _breakout_mixed(tbx, oracle_mod, n, seed):
    """covered states (worn walls, several balls, moved / resized paddles, multi-digit scores) mixed with states the direct
    kernel hands to the tile kernel: a custom brick table (i % 11 == 3), a ball in the HUD rows (i % 13 == 4), score digits
    clipped by the frame (123456789)"""
    pool, ref = _advance(tbx, oracle_mod, "breakout", n, 300, seed)
    rng = np.random.default_rng(seed)
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
        js["score"] = int(rng.choice([0, 7, 42, 860, 123456, 123456789]))
        js["lives"] = int(rng.choice([5, 1, 13]))
        if i % 11 == 3:
            js["bricks"][int(rng.integers(108))]["position"]["x"] += 3.0
        if i % 13 == 4:
            js["balls"] = [{"position": {"x": 100.0, "y": 5.0}, "velocity": {"x": 1.0, "y": 1.0}}]
        ref.write_state_json(i, js)
        states.append(js)
    pool.write_state_json(states)
    return pool, ref


def _amidar_painted(tbx, oracle_mod, n, seed):
    """painted corridors and boxes, moved / removed / caught enemies, checkerboard damage, multi-digit HUD values; a player
    inside the HUD rows (i % 10 == 1) makes the env one the direct kernel hands to the tile kernel"""
    pool, ref = _advance(tbx, oracle_mod, "amidar", n, 60, seed)
    rng = np.random.default_rng(seed)
    states = []
    for i in range(n):
        js = ref.state_json(i)
        tiles = js["board"]["tiles"]
        for _ in range(2 + i % 30):
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
            if i % 10 == 1:
                js["player"]["position"] = {"x": 960, "y": 2720}          # drawn on rows 206-212, the HUD's
        if i % 5 == 2:
            js["enemies"] = js["enemies"][:2]
            js["enemies"][0]["caught"] = True
            js["score"], js["lives"], js["jumps"] = int(rng.integers(0, 99999)), int(rng.integers(0, 20)), int(rng.integers(0, 10))
        if i % 5 == 3:
            for row in tiles[::3]:
                for x in range(0, 32, 2):
                    row[x] = "Empty" if row[x] != "Empty" else "Unpainted"
        ref.write_state_json(i, js)
        states.append(js)
    pool.write_state_json(states)
    return pool, ref


def _si_adversarial(tbx, oracle_mod, n, seed):
    """sprites clipped by the frame, invaders on top of each other / of shields / of lasers, huge lasers, eroded and moved
    shields, recoloured ship (no patch set), ufo, explosions, lives display, packed invaders"""
    pool, ref = _advance(tbx, oracle_mod, "space_invaders", n, 300, seed)
    rng = np.random.default_rng(seed)
    states = []
    for i in range(n):
        js = ref.state_json(i)
        k = i % 10
        if k == 1:
            for e in js["enemies"][:8]:
                e["x"], e["y"] = int(rng.integers(-12, 316)), int(rng.integers(-8, 205))
        elif k == 2:
            for e in js["enemies"][6:18]:
                e["x"], e["y"] = js["shields"][0]["x"] + int(rng.integers(-10, 10)), js["shields"][0]["y"] + int(rng.integers(-8, 12))
        elif k == 3:
            js["enemy_lasers"] = [{"x": int(rng.integers(0, 318)), "y": int(rng.integers(0, 190)), "w": 2, "h": 8, "t": 0, "movement": "Down", "speed": 3,
                                   "color": {"r": 252, "g": 252, "b": 84, "a": 255}} for _ in range(4)]
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
            js["ufo"]["appearance_counter"] = None
            js["ufo"]["death_counter"] = 9
            js["ship"]["alive"] = False
            js["ship"]["death_counter"] = 12
        elif k == 9:
            for j, e in enumerate(js["enemies"]):
                e["x"], e["y"] = 40 + 17 * (j % 12), 30 + 11 * (j // 12)
        ref.write_state_json(i, js)
        states.append(js)
    pool.write_state_json(states)
    return pool, ref


# ------------------------------------------------------------------------------------------------ A. multi-chunk walks
GRIDS = ["1", "2", "3", "7", None]
# per game: three sizes the direct kernel covers (Amidar and Space Invaders are not covered at 64 x 64: more than 4 taps per
# output row; 128 x 128 and 92 x 83 take their place -- 92 x 83 is a Space Invaders size without sprite patch tables)
A_SIZES = {"breakout": [(84, 84), (96, 80), (64, 64)], "amidar": [(84, 84), (96, 80), (128, 128)],
           "space_invaders": [(84, 84), (96, 80), (92, 83)]}
A_POOLS = {"breakout": (_breakout_mixed, 203), "amidar": (_amidar_painted, 99), "space_invaders": (_si_adversarial, 101)}


@pytest.mark.parametrize("game", ["breakout", "amidar", "space_invaders"])
def test_direct_kernel_multi_chunk_schedule(tbx, oracle_mod, game):
    """Ragged mixed pools (Breakout 203 envs = 51 team chunks of 4, Amidar 99, Space Invaders 101) rendered with persistent
    grids of 1, 2, 3 and 7 CTAs and the default grid.  With TBX_DIRECT_GRID=1 one CTA's two teams walk every chunk and fill
    the hand-over list alone.  Every size is rendered twice in a row, and the size and grid change between renders in a
    rotating order: the chunk counter and the hand-over list must be re-armed whatever the previous launch was.  Then 20
    frames are stepped and everything is repeated once."""
    build, n = A_POOLS[game]
    sizes = A_SIZES[game]
    for size in sizes:
        _covered(game, size)
    pool, ref = build(tbx, oracle_mod, n, 5)
    try:
        for rnd in range(2):
            for gi, grid in enumerate(GRIDS):
                _set({} if grid is None else {"TBX_DIRECT_GRID": grid})
                for k in range(len(sizes)):
                    size = sizes[(k + gi) % len(sizes)]
                    for rep in range(2):
                        _render_check(pool, ref, n, size, "%s round %d grid %s render %d" % (game, rnd, grid or "default", rep))
            _set({})
            _step(pool, ref, oracle_mod, game, n, 20, 1000 * rnd)
        pool.check()
    finally:
        _set({})
        pool.close()


# --------------------------------------------------------------------------------- B. a hand-over list of many chunks
def test_handover_list_longer_than_tile_grid(tbx, oracle_mod):
    """3,000 Breakout envs of which 2,500 are handed over by the direct kernel (a custom brick table, or a ball inside the
    HUD rows): more than 296 CTAs x 8 list entries, so the env-list tile kernel's loop takes a second pass.  The states are
    64 advanced games, written with per-env edits into every env of both the pool and the oracle."""
    m, n = 64, 3000
    src_pool, src = _advance(tbx, oracle_mod, "breakout", m, 300, 9)
    src_pool.close()
    base = [src.state_json(i) for i in range(m)]
    pool = tbx.BatchedToybox("breakout", n, seeds=9)
    ref = oracle_mod.OracleBatch("breakout", n, seeds=9 + np.arange(n))
    rng = np.random.default_rng(9)
    states = []
    n_handed = 0
    for i in range(n):
        js = copy.deepcopy(base[i % m])
        for k in rng.choice(108, size=int(rng.integers(0, 60)), replace=False):
            js["bricks"][int(k)]["alive"] = False
        js["score"] = int(rng.choice([0, 7, 42, 860, 123456]))
        kind = i % 6
        if kind in (1, 3, 5):                   # custom brick table: one of 108 shifted bricks
            js["bricks"][i % 108]["position"]["x"] += 2.0
        elif kind in (2, 4):                    # a ball inside the HUD rows
            js["balls"] = [{"position": {"x": float(rng.uniform(10, 230)), "y": float(rng.uniform(2, 9))}, "velocity": {"x": 1.0, "y": 1.0}}]
        n_handed += kind != 0
        ref.write_state_json(i, js)
        states.append(js)
    pool.write_state_json(states)
    assert n_handed >= 2500 and n_handed > 296 * 8
    e = emu_lib.Emu("breakout")
    for i in range(12):                          # the host restatement of the direct kernel hands over exactly kinds 1..5
        e.write_state_json(states[i])
        assert (e.render_direct() is None) == (i % 6 != 0), i
    try:
        for grid in (None, "1"):
            _set({} if grid is None else {"TBX_DIRECT_GRID": grid})
            for size in ((84, 84), (96, 80)):
                for rep in range(2):
                    _render_check(pool, ref, n, size, "grid %s render %d" % (grid or "default", rep))
        pool.check()
    finally:
        _set({})
        pool.close()


# ------------------------------------------------------------------------------------------- C. edited configs
def _col(r, g, b):
    return {"r": r, "g": g, "b": b, "a": 255}


def _brk_cfg(rows=6, **edit):
    cfg = emu_lib.Emu("breakout").config_json()
    cfg["row_colors"] = (cfg["row_colors"] * 2)[:rows]
    cfg["row_scores"] = (cfg["row_scores"] * 2)[:rows]
    cfg.update(edit)
    return cfg


def _ami_board():
    """the default board with two dangling stubs added to the track"""
    board = [list(r) for r in emu_lib.Emu("amidar").config_json()["board"]]
    for y in range(1, 4):
        board[y][3] = "="
    for x in range(8, 12):
        board[19][x] = "="
    return ["".join(r) for r in board]


def _config(game, name):
    """the edited configs, built from the game's defaults; a row colour of "row_luma_bg" is (0, 0, 1): gray 0, the
    black background's"""
    if game == "breakout":
        return {"rows1": lambda: _brk_cfg(1), "rows4": lambda: _brk_cfg(4), "rows8": lambda: _brk_cfg(8),
                "frame_is_bg": lambda: _brk_cfg(frame_color=_col(0, 0, 0)),
                "row_luma_bg": lambda: _brk_cfg(row_colors=[_col(200, 72, 72), _col(0, 0, 1), _col(180, 122, 48), _col(162, 162, 42),
                                                            _col(72, 160, 72), _col(66, 72, 200)]),
                "paddle_ball": lambda: _brk_cfg(paddle_color=_col(30, 200, 250), ball_color=_col(250, 250, 250))}[name]()
    cfg = emu_lib.Emu(game).config_json()
    edit = {"six_colours": dict(bg_color=_col(20, 30, 40), unpainted_color=_col(10, 120, 220), painted_color=_col(240, 30, 30),
                                inner_painted_color=_col(30, 200, 90), player_color=_col(250, 250, 250), enemy_color=_col(90, 60, 250)),
            "two_looks_one_gray": dict(painted_color=_col(148, 0, 211)),          # painted track in the unpainted colour
            "enemy_is_painted": dict(enemy_color=_col(255, 255, 30)),
            "board": {"board": _ami_board()} if game == "amidar" else None,
            "default": {},
            "shields": dict(shields=[[60, 157], [150, 150], [236, 160]])}[name]
    cfg.update(edit)
    return cfg


BRK_CONFIGS = {"rows1": 1, "rows4": 4, "rows8": 8, "frame_is_bg": 6, "row_luma_bg": 6, "paddle_ball": 6}   # name: brick rows
AMI_CONFIGS = ["six_colours", "two_looks_one_gray", "enemy_is_painted", "board"]
SI_CONFIGS = ["default", "shields"]
C_SIZES = {"breakout": [(84, 84), (96, 80), (64, 64), (128, 128)], "amidar": [(84, 84), (96, 80), (128, 128), (92, 83)],
           "space_invaders": [(84, 84), (92, 76), (92, 83), (128, 128)]}
# Space Invaders: sprite patch tables at 84 x 84 and 92 x 76 (80 x 105 phases), none at 92 x 83 (80 x 210 phases: over the
# tables' 4 MB) and 128 x 128.  Every size the direct kernel accepts has the score strip (see test_direct_area.py's table)
SI_PATCHES = {(84, 84): 12, (92, 76): 12, (92, 83): 0, (128, 128): 0}


def _advance_cfg(tbx, oracle_mod, game, cfg, n, steps, seed):
    """_advance with a config: the tracking policy for Breakout, random play for the others"""
    pool = tbx.BatchedToybox(game, n, seeds=seed, config=cfg)
    ref = oracle_mod.OracleBatch(game, n, seeds=seed + np.arange(n), cfg_json=cfg)
    legal = np.asarray(oracle_mod.LEGAL[game], np.int32)
    for t in range(steps):
        acts = legal[[oracle_mod.action_index(0xB200, i, t, len(legal)) for i in range(n)]]
        if game == "breakout":
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


def _edit_breakout(js, i, rng, nrows):
    bricks = js["bricks"]
    if i % 4 == 1:                               # whole brick rows dead (bricks are column-major: row = index % rows)
        dead = set(rng.choice(nrows, size=max(1, nrows // 2), replace=False).tolist())
        for k, b in enumerate(bricks):
            if k % nrows in dead:
                b["alive"] = False
    elif i % 4 == 2:                             # everything but one row dead, several balls inside the wall
        keep = int(rng.integers(nrows))
        for k, b in enumerate(bricks):
            b["alive"] = k % nrows == keep
        js["balls"] = [{"position": {"x": bricks[k]["position"]["x"] + 3.0, "y": bricks[k]["position"]["y"] + 1.0}, "velocity": {"x": 1.0, "y": 1.0}}
                       for k in rng.choice(len(bricks), size=3, replace=False).tolist()]
    elif i % 4 == 3:
        for k in rng.choice(len(bricks), size=int(rng.integers(0, len(bricks))), replace=False):
            bricks[int(k)]["alive"] = False
        js["paddle_width"] = float(rng.choice([48.0, 7.0]))
    js["score"] = int(rng.choice([0, 7, 860, 123456]))


def _edit_amidar(js, i, rng):
    tiles = js["board"]["tiles"]
    for _ in range(3 + i):
        ty, tx, ln, horiz = int(rng.integers(31)), int(rng.integers(32)), int(rng.integers(1, 20)), bool(rng.integers(2))
        for k in range(ln):
            y, x = (ty, tx + k) if horiz else (ty + k, tx)
            if y < 31 and x < 32 and tiles[y][x] in ("Unpainted", "ChaseMarker"):
                tiles[y][x] = "Painted"
    for b in js["board"]["boxes"][: i % 9]:
        b["painted"] = True


def _edit_si(js, i, rng):
    if i % 3 == 1:
        for sh in js["shields"]:
            for row in sh["data"]:
                for c in rng.choice(16, size=5, replace=False):
                    row[int(c)] = {"r": 0, "g": 0, "b": 0, "a": 0}
    elif i % 3 == 2:
        for j, e in enumerate(js["enemies"]):
            e["x"], e["y"] = 40 + 17 * (j % 12), 30 + 11 * (j // 12)
        js["score"] = int(rng.choice([35, 1250, 99999]))


def _config_case(tbx, oracle_mod, game, name, n=24):
    cfg = _config(game, name)
    sizes = C_SIZES[game]
    for size in sizes:
        info = _covered(game, size, cfg)
        if game == "breakout":
            assert info["nrows"] == BRK_CONFIGS[name], (name, size, info)
        if game == "space_invaders":
            assert (info["n_sets"], info["sc_ok"]) == (SI_PATCHES[size], 1), (name, size, info)
    pool, ref = _advance_cfg(tbx, oracle_mod, game, cfg, n, 300 if game == "breakout" else 120, 31)
    rng = np.random.default_rng(17)
    states = []
    for i in range(n):
        js = ref.state_json(i)
        if game == "breakout":
            _edit_breakout(js, i, rng, len(cfg["row_colors"]))
        elif game == "amidar":
            _edit_amidar(js, i, rng)
        else:
            _edit_si(js, i, rng)
        ref.write_state_json(i, js)
        states.append(js)
    pool.write_state_json(states)
    try:
        for rnd in range(2):
            for size in sizes:
                for v in ({}, TILE):
                    _set(v)
                    _render_check(pool, ref, n, size, "%s config %s round %d %s" % (game, name, rnd, v or "direct"))
            _set({})
            if rnd == 0:
                for mode in ("rgb", "rgba", "gray"):
                    want = ref.render(mode).reshape(n, -1)
                    got = pool.render(obs=mode).cpu().numpy().reshape(n, -1)
                    _assert_same(got[:, None], want[:, None], "%s config %s %s" % (game, name, mode))
                _step(pool, ref, oracle_mod, game, n, 30, 700)
        pool.check()
    finally:
        _set({})
        pool.close()


@pytest.mark.parametrize("name", list(BRK_CONFIGS))
def test_breakout_config_through_direct_kernel(tbx, oracle_mod, name):
    """brick-row counts 1 / 4 / 8 (8 rows = 144 bricks, the record's capacity; the kernel's shared H look-up rows and row
    masks follow the count), the frame in the background colour, a row whose gray equals the background's, and recoloured
    paddle and ball -- with whole rows dead and balls inside the wall"""
    _config_case(tbx, oracle_mod, "breakout", name)


@pytest.mark.parametrize("name", AMI_CONFIGS)
def test_amidar_config_through_direct_kernel(tbx, oracle_mod, name):
    """all six colours changed, painted and unpainted track of one gray, enemies in the painted colour, and an edited
    config board (build_ami_direct takes the board's looks from the config, so an edited board is covered)"""
    _config_case(tbx, oracle_mod, "amidar", name)


@pytest.mark.parametrize("name", SI_CONFIGS)
def test_space_invaders_config_through_direct_kernel(tbx, oracle_mod, name):
    """moved shields (they are part of the base frame) and the default config, at sizes with sprite patch tables (84 x 84,
    92 x 76) and without (92 x 83, 128 x 128), each with the score strip.  No size the direct kernel accepts lacks the
    strip, so that combination cannot be rendered (test_direct_area.py checks this over every accepted size)."""
    _config_case(tbx, oracle_mod, "space_invaders", name)


# ------------------------------------------------------------------------------------ D. dual tile kernel (wrapped)
# sizes the dual kernel accepts (at most 5 x 4 taps; 64 x 64 and 48 x 60 are over that for Amidar and Space Invaders)
D_SIZES = {"breakout": [(84, 84), (64, 64), (48, 60)], "amidar": [(84, 84), (96, 80), (128, 128)],
           "space_invaders": [(84, 84), (96, 80), (92, 76)]}
D_VARIANTS = [{"TBX_AREA_LCAP": "3"}, {"TBX_AREA_LCAP": "24"}, {}, {"TBX_AREA_DIGIT_CACHE": "0"},
              {"TBX_AREA_LCAP": "3", "TBX_AREA_DIGIT_CACHE": "0"}]


def _intervene(game, js, i, rng):
    if game == "breakout":                       # many dead bricks, 2-4 balls, a wide paddle
        for k in rng.choice(108, size=int(rng.integers(40, 100)), replace=False):
            js["bricks"][int(k)]["alive"] = False
        js["balls"] = [{"position": {"x": float(rng.uniform(20, 220)), "y": float(rng.uniform(40, 130))},
                        "velocity": {"x": float(rng.choice([-2.0, 2.0])), "y": float(rng.choice([-2.0, 2.0]))}} for _ in range(2 + i % 3)]
        js["paddle_width"] = 48.0
    elif game == "space_invaders":               # packed invaders, lasers, eroded shields
        for j, e in enumerate(js["enemies"]):
            e["x"], e["y"] = 40 + 17 * (j % 12), 40 + 11 * (j // 12)
        js["enemy_lasers"] = [{"x": int(rng.integers(20, 300)), "y": int(rng.integers(60, 150)), "w": 2, "h": 8, "t": 0, "movement": "Down", "speed": 3,
                               "color": {"r": 252, "g": 252, "b": 84, "a": 255}} for _ in range(3)]
        for sh in js["shields"]:
            for row in sh["data"]:
                for c in rng.choice(16, size=6, replace=False):
                    row[int(c)] = {"r": 0, "g": 0, "b": 0, "a": 0}
    else:                                        # painted corridors and boxes
        tiles = js["board"]["tiles"]
        for _ in range(6 + 2 * i):
            ty, tx, ln, horiz = int(rng.integers(31)), int(rng.integers(32)), int(rng.integers(1, 20)), bool(rng.integers(2))
            for k in range(ln):
                y, x = (ty, tx + k) if horiz else (ty + k, tx)
                if y < 31 and x < 32 and tiles[y][x] in ("Unpainted", "ChaseMarker"):
                    tiles[y][x] = "Painted"
        for b in js["board"]["boxes"][: 2 + i % 6]:
            b["painted"] = True


def _run_dual(game, n, size, steps, seed0=600):
    import torch
    from oracle import oracle as O
    from oracle import wrappers as OW
    from toybox_b200.wrappers import DeepmindToybox
    env = DeepmindToybox(game, n, seeds=seed0, noop_seed=7, size=size)
    refs = [OW.WrappedEnv(game, seed0 + i, env_id=i, noop_seed=7, size=size) for i in range(n)]
    rng = np.random.default_rng(seed0)
    try:
        obs = env.reset()
        want = np.stack([r.reset() for r in refs])
        _assert_same(obs[:, env.order()].cpu().numpy().reshape(n, -1, size[0]), want.reshape(n, -1, size[0]), "%s %s reset" % (game, size))
        for t in range(steps):
            if t == 3:                           # the same adversarial states on both sides
                states = []
                for i, r in enumerate(refs):
                    js = r.base.b.state_json(0)
                    _intervene(game, js, i, rng)
                    r.base.b.write_state_json(0, js)
                    states.append(js)
                env.pool.write_state_json(states)
            v = D_VARIANTS[(t // 2) % len(D_VARIANTS)]
            _set(v)
            acts = np.asarray([O.action_index(0xB200, i, t, env.n_actions) for i in range(n)], np.int32)
            obs, rew, done, info = env.step(torch.as_tensor(acts, device=env.device))
            got = obs[:, env.order()].cpu().numpy()
            rew, done, lives = rew.cpu().numpy(), done.cpu().numpy().astype(bool), info["lives"].cpu().numpy()
            wants = []
            for i, r in enumerate(refs):
                w_obs, w_rew, w_done, w_info = r.step(int(acts[i]))
                assert (w_rew, w_done, w_info["lives"]) == (rew[i], done[i], lives[i]), (game, size, t, i, v, w_rew, rew[i], w_done, done[i])
                wants.append(w_obs)
            want = np.stack(wants)
            _assert_same(got.reshape(n, -1, size[0]), want.reshape(n, -1, size[0]), "%s %s step %d variant %s" % (game, size, t, v))
        env.check()
    finally:
        _set({})
        env.close()


@pytest.mark.parametrize("game", ["breakout", "amidar", "space_invaders"])
def test_dual_tile_kernel_overflow_and_interventions(game):
    """DeepmindToybox against oracle.wrappers.WrappedEnv env by env (stacked observations, rewards, dones, lives) at three
    sizes per game, with adversarial states written into both after three agent steps, while the list capacity cycles
    through 3, 24 and the default and the digit patches are switched off: the dual list sweep, the per-tile rebuild and the
    both-frames flag of every run.

    redo_all (the two frames on different base frames) is not reachable through the wrapper: only Breakout has two base
    frames, an env's base frame changes only with its brick table, and the table changes only at new_game or at a state
    write.  A state write happens between agent steps, and every agent step copies the state into the second frame after
    its last new_game (the no-op unit of a reset always snapshots; a skip unit snapshots before its last frame, which does
    not change the table).  So both frames of an observation always share the table."""
    for k, size in enumerate(D_SIZES[game]):
        info = emu_lib.Emu(game).direct_info(*size)
        assert info["taps"][0] <= 5 and info["taps"][1] <= 4, (game, size, info)
        _run_dual(game, 6, size, 24, seed0=600 + 10 * k)


def test_dual_tile_kernel_refuses_many_tap_sizes():
    """wrapped observations need the 5 x 4 tile kernel: Breakout 100 x 37 (4 x 6 taps) is refused with the library's error"""
    from toybox_b200 import _lib
    from toybox_b200.wrappers import DeepmindToybox
    assert emu_lib.Emu("breakout").direct_info(100, 37)["taps"] == (4, 6)
    with pytest.raises(_lib.ToyboxError, match="wrapped observations need an output size"):
        env = DeepmindToybox("breakout", 4, seeds=1, size=(100, 37))
        try:
            env.reset()
        finally:
            env.close()
