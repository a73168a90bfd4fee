"""CPU tier: the DIRECT INTER_AREA algorithm of the Breakout kernel (tbx_direct.h: wall rows from look-up tables, movers
evaluated tap by tap, HUD digit patches), emulated on the host from the same headers, equals the straightforward
full-frame resize -- over random and brick-breaking rollouts, interventions and other output sizes -- and hands exactly
the states it does not cover to the general kernel."""
import numpy as np
import pytest

import emu_lib


def _track(e, t, i=1):
    """ball-tracking action with a slowly varying aim error (breaks bricks, unlike the random stream)"""
    r = e.record()
    if r[63]:                                             # is_dead: serve
        return 1
    f = r.view(np.float64)
    bx, px = f[12] + (((i * 7 + t // 50) % 9) - 4), f[8]
    return 3 if bx > px + 1 else 4 if bx < px - 1 else 0


@pytest.mark.parametrize("policy", ["random", "track"])
def test_direct_equals_full_over_rollout(oracle_mod, policy):
    e = emu_lib.Emu("breakout")
    e.seed(31)
    e.new_game()
    legal = oracle_mod.LEGAL["breakout"]
    n_direct = 0
    max_dead = 0
    for t in range(9000 if policy == "track" else 3000):
        a = _track(e, t) if policy == "track" else legal[oracle_mod.action_index(11, 0, t, len(legal))]
        e.step(ale_action=a, auto_reset=True)
        if t % 23 == 0:
            d = e.render_direct()
            assert d is not None, t
            n_direct += 1
            assert np.array_equal(d, e.render("gray84")), t
            max_dead = max(max_dead, 108 - sum(bin(int(w)).count("1") for w in e.record()[66:71]))
    assert n_direct > 100
    if policy == "track":
        assert max_dead >= 30, max_dead              # the wall really got worn


def test_direct_interventions_and_sizes(oracle_mod):
    b = emu_lib.Emu("breakout")
    for t in range(300):
        b.step(ale_action=_track(b, t), auto_reset=True)
    js = b.state_json()
    rng = np.random.default_rng(3)
    for trial in range(30):
        s = dict(js)
        s["bricks"] = [dict(k) for k in js["bricks"]]
        for k in rng.choice(108, size=int(rng.integers(0, 108)), replace=False):
            s["bricks"][int(k)]["alive"] = False
        s["balls"] = [{"position": {"x": float(rng.uniform(0, 240)), "y": float(rng.uniform(20, 170))}, "velocity": {"x": 1.0, "y": 1.0}}
                      for _ in range(int(rng.integers(0, 5)))]
        s["paddle"] = dict(js["paddle"])
        s["paddle"]["position"] = {"x": float(rng.uniform(0, 240)), "y": float(rng.choice([143.0, 60.0, 50.5, 158.0]))}
        s["paddle_width"] = float(rng.choice([24.0, 24.0, 48.0, 7.0, 300.0]))
        s["ball_radius"] = float(rng.choice([2.0, 2.0, 5.5, 0.5]))
        s["score"] = int(rng.choice([0, 7, 42, 860, 123456, 123456789]))
        s["lives"] = int(rng.choice([5, 1, 0, 13]))
        b.write_state_json(s)
        for size in ((84, 84), (96, 80), (64, 64), (100, 37), (128, 128)):
            d = b.render_direct(*size)
            if size == (100, 37):                     # 5 taps per output row: outside the direct kernel's limits
                assert d is None
                continue
            if s["score"] == 123456789:               # digits clipped by the frame edge have no patch: the tile kernel's
                assert d is None
                continue
            assert d is not None, (trial, size)
            assert np.array_equal(d, b.render("gray84", *size)), (trial, size)
        assert b.render_direct(42, 42) is None        # output width not a multiple of 4: the tile kernel's


def test_direct_hands_over_what_it_does_not_cover(oracle_mod):
    b = emu_lib.Emu("breakout")
    js = b.state_json()
    s = dict(js)
    s["balls"] = [{"position": {"x": 100.0, "y": 5.0}, "velocity": {"x": 1.0, "y": 1.0}}]       # a ball inside the HUD rows
    b.write_state_json(s)
    assert b.render_direct() is None
    s = dict(js)
    s["bricks"] = [dict(k) for k in js["bricks"]]
    s["bricks"][3]["position"] = {"x": 15.0, "y": 43.0}                                         # custom brick table
    b.write_state_json(s)
    assert b.render_direct() is None
    b.write_state_json(js)
    assert np.array_equal(b.render_direct(), b.render("gray84"))
    cfg = b.config_json()
    cfg["bg_color"] = {"r": 40, "g": 50, "b": 60, "a": 255}
    cfg["frame_color"] = {"r": 200, "g": 10, "b": 10, "a": 255}
    cfg["row_colors"] = cfg["row_colors"][:4]
    cfg["row_scores"] = cfg["row_scores"][:4]
    b.write_config_json(cfg)
    b.new_game()
    for t in range(600):
        b.step(ale_action=_track(b, t), auto_reset=True)
    assert np.array_equal(b.render_direct(), b.render("gray84"))


@pytest.mark.parametrize("size", [(84, 84), (96, 80), (64, 64), (48, 60), (128, 128)])
def test_si_score_strip_table_equals_full_resize(size):
    """Space Invaders: the score rendered as one strip from the host-built table of digit pairs (TbxSiDirect.sc_px, the direct kernel's
    step 2c, emulated on the host) equals the full-frame resize for scores that put every pair of digits (and the empty slot) next
    to each other at every position, single digits and ten-digit scores."""
    scores = [0, 7, 10, 99, 100, 101, 909, 1000, 4711, 99999, 1234567, 98765432, 123456789, 999999999, 1000000000, 1999999999, 2147483647]
    for k in range(9):
        for a in range(10):
            for b in range(10):
                v = a * 10 ** k + b * 10 ** (k + 1) + (10 ** (k + 2) if b == 0 and k + 2 <= 9 else 0)
                if 0 < v <= 2147483647:
                    scores.append(v)
    e = emu_lib.Emu("space_invaders")
    e.seed(5)
    e.new_game()
    js = e.state_json()
    ow, oh = size
    n_table = 0
    for v in sorted(set(scores)):
        js["score"] = int(v)
        e.write_state_json(js)
        want = e.render("gray84", ow, oh)
        got = e.si_score_strip(ow, oh)
        if got is None:
            continue
        n_table += 1
        bad = np.argwhere(got != want)
        assert bad.size == 0, (size, v, bad[:4], got[tuple(bad[0])], want[tuple(bad[0])])
    assert n_table > 0 or size != (84, 84)          # the table exists at the size the benchmark uses


def test_direct_coverage_of_gpu_tier_cases():
    """The direct kernels' tables exist for every (config, output size) that test_gpu_area_coverage.py renders through them,
    with the brick rows and Space Invaders sprite patch sets it claims, and the wrapped sizes it uses stay within the dual
    tile kernel's 5 x 4 taps.  Over every output size the library accepts, Space Invaders' direct kernel runs both with and
    without sprite patch tables but always with the score strip.  A builder change that drops coverage fails here."""
    import test_gpu_area_coverage as G
    for game, sizes in G.A_SIZES.items():
        for size in sizes:
            assert emu_lib.Emu(game).direct_info(*size)["ok"] == 1, (game, size)
    for game, names in (("breakout", list(G.BRK_CONFIGS)), ("amidar", G.AMI_CONFIGS), ("space_invaders", G.SI_CONFIGS)):
        for name in names:
            e = emu_lib.Emu(game, G._config(game, name))
            for size in G.C_SIZES[game]:
                info = e.direct_info(*size)
                assert info["ok"] == 1, (game, name, size, info)
                if game == "breakout":
                    assert info["nrows"] == G.BRK_CONFIGS[name], (name, size, info)
                if game == "space_invaders":
                    assert (info["n_sets"], info["sc_ok"]) == (G.SI_PATCHES[size], 1), (name, size, info)
    for game, sizes in G.D_SIZES.items():
        for size in sizes:
            tx, ty = emu_lib.Emu(game).direct_info(*size)["taps"]
            assert tx <= 5 and ty <= 4, (game, size, tx, ty)
    e = emu_lib.Emu("space_invaders")
    seen = set()
    for w in range(4, 129, 4):                   # the direct kernel needs a width that is a multiple of 4
        for h in range(1, 129):
            try:
                info = e.direct_info(w, h)
            except ValueError:                   # a size the library refuses
                continue
            if info["ok"]:
                seen.add((info["n_sets"] > 0, info["sc_ok"]))
    assert seen == {(True, 1), (False, 1)}, seen
