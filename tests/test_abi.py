"""CPU tier: the C-ABI library builds for sm_100a, loads, and exports every symbol include/toybox_b200.h declares.
No compute calls (no GPU here)."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "toybox_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(tbx_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_loads_and_exports_every_declared_symbol():
    import toybox_b200
    toybox_b200.build()
    L = toybox_b200.lib()
    names = declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(L, n), n
    assert sorted(toybox_b200._lib.SIGNATURES) == names
    assert toybox_b200._lib.EXPORTS == names
    assert L.tbx_version() >= 100


def test_no_cpu_fallback_without_a_gpu():
    import torch
    import toybox_b200
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(toybox_b200.ToyboxError):
        toybox_b200.BatchedToybox("breakout", 4)
    out = C.c_void_p()
    rc = toybox_b200.lib().tbx_pool_create(b"breakout", 4, 0, None, C.byref(out))
    assert rc != 0 and not out.value and b"no CPU path" in toybox_b200.lib().tbx_last_error()


def test_host_only_entry_points_work_without_a_gpu():
    import toybox_b200
    sch = toybox_b200.schema_for_state("amidar")
    assert "board" in sch["required"]
    assert "jitter" in toybox_b200.schema_for_config("space_invaders")["required"]
    out = C.c_void_p()
    assert toybox_b200.lib().tbx_pool_create(b"pong", 4, 0, None, C.byref(out)) != 0


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "toybox_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".h", ".cu", ".cuh", ".cpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle|oracle/|oracle\.py|tbo\.h", text, flags=re.M), (dirpath, f)
                assert "libtbo" not in text and "tbo_" not in text, (dirpath, f)


def test_field_lookup_is_host_only_and_matches_the_record_layout():
    """tbx_field_lookup (SURVEY 8 f3) needs no GPU: property paths of the JSON state schema -> (word, kind, bit)"""
    import ctypes as C
    from toybox_b200 import _lib
    L = _lib.lib()

    def look(game, path):
        w, k, b = C.c_int(-1), C.c_int(-1), C.c_int(-1)
        rc = L.tbx_field_lookup(game.encode(), path.encode(), C.byref(w), C.byref(k), C.byref(b))
        return rc, w.value, k.value, b.value

    # header words: rand[2] u64, sim_rand[2] u64 = words 0..7, then lives, score, level
    for game in ("breakout", "amidar", "space_invaders"):
        assert look(game, "lives")[:3] == (0, 8, 0) and look(game, "score")[:3] == (0, 9, 0) and look(game, "level")[:3] == (0, 10, 0)
    rc, w, k, b = look("breakout", "paddle.position.x")
    assert rc == 0 and w == 16 and k == 1                      # the first f64 after the 16-word header
    assert look("breakout", "paddle.velocity.y")[1] == 16 + 6
    rc, w0, k, b0 = look("breakout", "bricks[0].alive")
    rc, w37, k, b37 = look("breakout", "bricks[37].alive")
    assert k == 3 and b0 == 0 and w37 == w0 + 1 and b37 == 5   # bit 37 = word 1, bit 5 of the alive mask
    assert look("space_invaders", "ufo.appearance_counter")[2] == 4 and look("amidar", "board.boxes[28].painted")[2:] == (3, 28)
    assert look("amidar", "enemies[1].position.y")[1] - look("amidar", "enemies[0].position.y")[1] == 31   # AmiMob = 31 words
    for game, path in (("breakout", "no.such"), ("breakout", "balls[9].position.x"), ("amidar", "ship.x"), ("pong", "lives")):
        assert look(game, path)[0] != 0
        assert b"" != L.tbx_last_error()
