"""Runs the reference's OWN unit tests (test/interventions/*.py, scripts/utils/test_games.py logic) against a ctoybox
module backed by
  (a) the host build of the product's engines + JSON codec (tests/emu)            -- CPU tier
  (b) the oracle                                                                    -- CPU tier
  (c) the CUDA library itself, through toybox_b200.ctoybox.Toybox (batch of 1)      -- GPU tier
The reference's Python is the byte-identical snapshot tests/golden/reference_py/ (made by tests/golden/make_golden.py), so
that every tier runs the same files on any machine."""
import os
import sys
import types
import unittest

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(HERE, "golden", "reference_py")


def install_ctoybox(toybox_cls, input_cls):
    """Make `import ctoybox` resolve to a module whose Toybox is `toybox_cls`, and forget any loaded `toybox` package."""
    m = types.ModuleType("ctoybox")
    m.Toybox, m.Input, m.Simulator, m.State = toybox_cls, input_cls, object, object
    sys.modules["ctoybox"] = m
    for name in [k for k in sys.modules if k == "toybox" or k.startswith("toybox.") or k == "test" or k.startswith("test.")]:
        del sys.modules[name]
    return m


def run_reference_tests(toybox_cls, input_cls):
    install_ctoybox(toybox_cls, input_cls)
    if REF in sys.path:
        sys.path.remove(REF)
    sys.path.insert(0, REF)
    try:
        suite = unittest.defaultTestLoader.discover(os.path.join(REF, "test", "interventions"), top_level_dir=REF)
        return unittest.TextTestRunner(verbosity=0, stream=open(os.devnull, "w")).run(suite)
    finally:
        sys.path.remove(REF)
        sys.modules.pop("ctoybox", None)
        for name in [k for k in sys.modules if k == "toybox" or k.startswith("toybox.") or k == "test" or k.startswith("test.")]:
            del sys.modules[name]


def check(res):
    msgs = ["%s: %s" % (t.id(), tb.strip().splitlines()[-1]) for t, tb in res.failures + res.errors]
    assert res.testsRun >= 30, res.testsRun
    assert not msgs, "\n".join(msgs)


@pytest.mark.parametrize("backend", ["emu", "oracle"])
def test_reference_intervention_tests(backend):
    import shims
    from oracle import oracle as O
    check(run_reference_tests(shims.EmuToybox if backend == "emu" else shims.OracleToyboxWithSchema, O.Input))


@pytest.mark.gpu
def test_reference_intervention_tests_on_the_cuda_path(tbx):
    """the reference's 30+ intervention tests, unmodified, with ctoybox = toybox_b200.ctoybox (every call runs a kernel)"""
    from toybox_b200 import ctoybox
    check(run_reference_tests(ctoybox.Toybox, ctoybox.Input))


def _smoke_script_logic(make):
    """scripts/utils/test_games.py:5-41 restated: score 0, lives > 0, 100 NOOPs, frames, JSON round trips."""
    for game in ("breakout", "amidar", "space_invaders"):
        tb = make(game)
        for _ in range(3):
            assert tb.get_score() == 0 and tb.get_lives() > 0
            for _ in range(100):
                tb.apply_ale_action(0)
            assert tb.get_rgb_frame().shape == (tb.get_height(), tb.get_width(), 3)
            assert tb.get_score() == 0 and tb.get_lives() > 0
            cfg, st = tb.config_to_json(), tb.to_state_json()
            tb.set_seed(1234)
            tb.write_config_json(cfg)
            tb.write_state_json(st)
            assert tb.to_state_json() == st
            tb.new_game()


def test_reference_smoke_script_logic():
    import shims
    _smoke_script_logic(shims.EmuToybox)


@pytest.mark.gpu
def test_reference_smoke_script_logic_on_the_cuda_path(tbx):
    from toybox_b200 import ctoybox
    _smoke_script_logic(ctoybox.Toybox)


@pytest.mark.gpu
def test_amidar_tile_queries_on_the_cuda_path(tbx):
    """query_state_json('tile_to_world' / 'world_to_tile') (toybox/interventions/amidar.py:508-518) through the library"""
    from toybox_b200 import ctoybox
    tb = ctoybox.Toybox("amidar")
    for tx, ty in ((0, 0), (31, 15), (7, 30), (12, 6)):
        w = tb.query_state_json("tile_to_world", {"tx": tx, "ty": ty})      # [x, y]: WorldPoint(self, *result), amidar.py:508-510
        assert list(w) == [64 * tx, 80 * ty]
        t = tb.query_state_json("world_to_tile", {"x": w[0] + 63, "y": w[1] + 79})
        assert list(t) == [tx, ty]
    assert list(tb.query_state_json("world_to_tile", {"x": -1, "y": -1})) == [-1, -1]
    tb.close()
    b = ctoybox.Toybox("breakout")
    assert b.rstate.breakout_bricks_remaining() == 108 and b.rstate.breakout_channel_count() == 0
    b.close()
