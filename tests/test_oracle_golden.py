"""Pins the oracle (and the product's host-built engines) to everything the reference's fixtures and tests
pin for this path (SURVEY 8c / App. A): RNG algorithm and seeding lineage, complete initial states of the three
games, post-FIRE known answers, cv2 INTER_AREA outputs."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import emu_lib
from conftest import json_diff

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GAMES = ["breakout", "amidar", "space_invaders"]


def gold(name):
    return json.load(open(os.path.join(GOLD, name)))


def test_rng_known_answers(oracle_mod):
    kat = gold("rng_kat.json")
    L = oracle_mod.lib()
    g = oracle_mod.Rng()
    g.s[0], g.s[1] = kat["seed_state"]
    assert [L.tbo_rng_next_u64(C.byref(g)) for _ in range(6)] == kat["outputs"]
    assert [int(g.s[0]), int(g.s[1])] == kat["state_after_6"]
    L.tbo_rng_seed(C.byref(g), C.c_uint32(13))          # seed 13 = amidar/breakout default config rand
    assert [int(g.s[0]), int(g.s[1])] == kat["seed_state"]
    # the Breakout child rng is born from draws 3,4 of that lineage and consumes exactly two draws to pick start #2 of 4
    g.s[0], g.s[1] = kat["breakout_child_born"]
    assert L.tbo_rng_index(C.byref(g), 4) == 2
    g.s[0], g.s[1] = kat["breakout_child_born"]
    assert [L.tbo_rng_next_u64(C.byref(g)) for _ in range(2)] == kat["breakout_child_draws"]


def strip_fixture_era(game, fx):
    """Map the (older-schema) fixture onto the 0.5.0-era key set the intervention classes require (SURVEY App. A.0)."""
    fx = json.loads(json.dumps(fx))
    if game == "breakout":
        fx["score"] = fx.pop("points")
        fx["level"] = 1
    elif game == "amidar":
        fx["level"] = 1
    else:
        e0 = fx["enemies"][0]
        fx["enemies_movement"] = {"move_counter": e0["move_counter"], "move_dir": "Right" if e0["move_right"] else "Left",
                                  "visual_orientation": e0["orientation_init"]}
        for e in fx["enemies"]:
            for k in ("move_down", "move_right", "orientation_init", "move_counter"):
                e.pop(k)
        fx["level"] = fx.pop("levels_completed") + 1
    return fx


def normalise_sets(game, js):
    if game == "amidar":       # box / junction order in the fixture is hash-set iteration order: compare as sets
        js = json.loads(json.dumps(js))
        js["board"]["boxes"] = sorted(js["board"]["boxes"], key=lambda b: (b["top_left"]["ty"], b["top_left"]["tx"]))
        js["board"]["junctions"] = sorted(js["board"]["junctions"])
        js["board"]["chase_junctions"] = sorted(js["board"]["chase_junctions"])
    return js


@pytest.mark.parametrize("game", GAMES)
@pytest.mark.parametrize("impl", ["oracle", "emu"])
def test_initial_state_equals_reference_fixture(oracle_mod, game, impl):
    want = normalise_sets(game, strip_fixture_era(game, gold("%s_state_default.json" % game)))
    got = oracle_mod.OracleToybox(game).to_state_json() if impl == "oracle" else emu_lib.Emu(game).state_json()
    assert json_diff(normalise_sets(game, got), want) == []


@pytest.mark.parametrize("game", GAMES)
@pytest.mark.parametrize("impl", ["oracle", "emu"])
def test_config_equals_reference_fixture(oracle_mod, game, impl):
    want = gold("%s_config_default.json" % game)
    tb = oracle_mod.OracleToybox(game)
    got = tb.config_to_json() if impl == "oracle" else emu_lib.Emu(game).config_json()
    if game != "amidar":       # breakout / space invaders dump the config rand after the constructor's new_game()s
        assert got["rand"] == want["rand"] or impl == "emu"
    got = dict(got, rand=want["rand"])
    assert json_diff(got, want) == []


@pytest.mark.parametrize("impl", ["oracle", "emu"])
def test_fixture_era_state_import(oracle_mod, impl):
    """The importer accepts the fixtures as they are (older key set) and reproduces the same state."""
    for game in GAMES:
        fx = gold("%s_state_default.json" % game)
        if impl == "oracle":
            tb = oracle_mod.OracleToybox(game)
            tb.write_state_json(fx)
            got = tb.to_state_json()
        else:
            e = emu_lib.Emu(game)
            e.write_state_json(fx)
            got = e.state_json()
        assert json_diff(normalise_sets(game, got), normalise_sets(game, strip_fixture_era(game, fx))) == []


@pytest.mark.parametrize("impl", ["oracle", "emu"])
def test_post_fire_known_answers(oracle_mod, impl):
    """test_breakout_interventions.py:141-142 (paddle (120,143)), :95 (>=1 ball); test_amidar_interventions.py:39,81,173."""
    def make(game):
        if impl == "oracle":
            tb = oracle_mod.OracleToybox(game)
            inp = oracle_mod.Input()
            inp.button1 = True
            tb.apply_action(inp)
            return tb.to_state_json()
        e = emu_lib.Emu(game)
        e.step(input_mask=16)
        return e.state_json()
    b = make("breakout")
    assert b["paddle"]["position"] == {"x": 120.0, "y": 143.0} and len(b["balls"]) >= 1 and len(b["bricks"]) == 108
    assert b["bricks"][1]["col"] == 0 and b["bricks"][1]["color"] != {"r": 72, "g": 72, "b": 72, "a": 72}
    a = make("amidar")
    assert a["board"]["tiles"][0][0] == "ChaseMarker" and len(a["enemies"]) == 5 and a["jumps"] == 3 and a["jump_timer"] > 0


def test_area_resize_equals_cv2_golden(oracle_mod):
    z = np.load(os.path.join(GOLD, "area_golden.npz"))
    L = oracle_mod.lib()
    for game, (w, h) in oracle_mod.DIMS.items():
        for kind, (dw, dh) in (("noise", (84, 84)), ("blocky", (84, 84)), ("noise_100x60", (100, 60))):
            src = np.ascontiguousarray(z["%s_src_%s" % (game, "noise" if kind.startswith("noise") else kind)])
            want = z["%s_dst_%s" % (game, kind)]
            got = np.empty((dh, dw), np.uint8)
            L.tbo_resize_area_u8(src.ctypes.data_as(C.c_void_p), w, h, 1, got.ctypes.data_as(C.c_void_p), dw, dh)
            assert np.array_equal(got, want), (game, kind)


def test_area_resize_equals_live_cv2(oracle_mod):
    """against cv2 itself where it is installed, and always against the digests of cv2's outputs for the same frames"""
    try:
        import cv2
    except ImportError:
        cv2 = None
    kat = gold("area_cv2_seed5.json")
    rng = np.random.default_rng(5)
    L = oracle_mod.lib()
    i = 0
    for (w, h) in oracle_mod.DIMS.values():
        for _ in range(5):
            src = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
            assert hashlib.sha256(src.tobytes()).hexdigest() == kat["src_sha256"][i], "numpy's seeded stream changed: regenerate the digests"
            got = np.empty((84, 84), np.uint8)
            L.tbo_resize_area_u8(src.ctypes.data_as(C.c_void_p), w, h, 1, got.ctypes.data_as(C.c_void_p), 84, 84)
            assert hashlib.sha256(got.tobytes()).hexdigest() == kat["dst_sha256"][i], (w, h, i)
            if cv2 is not None:
                assert np.array_equal(got, cv2.resize(src, (84, 84), interpolation=cv2.INTER_AREA))
            i += 1
