"""CPU tier: two shortcuts of the Breakout direct kernel (tbx_render_direct.cuh), checked on a host build of the same headers
(tests/emu/direct_check.cpp).

- brk_mover_rec reads the paddle and the balls straight from the record, with one saturating f64 -> int conversion and integer
  clamps, instead of building the draw-list primitive: it must give brk_mover's rectangle for every record, including the
  ones the game never produces (NaN, infinities, coordinates past the 2^29 saturation and the 16-bit clip, negative sizes).
- The kernel writes the HUD digit patches of its cached slots in one pass, in no particular order: that is only right when
  the patches of two cached slots never share an output pixel, at every output size the direct kernel accepts.
"""
import ctypes as C
import itertools
import os
import subprocess

import numpy as np
import pytest

import emu_lib

N_MOVERS = 5  # paddle + 4 balls
_HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """tests/emu/direct_check.cpp with the library's host half, built in a temporary directory"""
    so = str(tmp_path_factory.mktemp("direct_check") / "libdirect_check.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", so,
                           os.path.join(_HERE, "emu", "direct_check.cpp"),
                           os.path.join(os.path.dirname(_HERE), "toybox_b200", "csrc", "tbx_host.cpp")])
    lib = C.CDLL(so)
    lib.dc_brk_movers.argtypes = [C.c_void_p, C.c_void_p]
    lib.dc_brk_mover_words.argtypes = [C.c_void_p]
    lib.dc_digit_patch_boxes.argtypes = [C.c_int, C.c_int, C.c_void_p]
    return lib


def _words(L):
    out = np.zeros(6, np.int32)
    L.dc_brk_mover_words(out.ctypes.data_as(C.c_void_p))
    return dict(zip(("paddle_px", "paddle_py", "paddle_width", "ball_radius", "n_balls", "ball"), (int(v) for v in out)))


def _movers(L, rec):
    rec = np.ascontiguousarray(rec, np.uint32)
    out = np.zeros((N_MOVERS + 2, 10), np.int32)
    assert L.dc_brk_movers(rec.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)) == 0
    return out[:, :5], out[:, 5:]


def _set_f64(rec, w, v):
    rec[w:w + 2] = np.array([v], np.float64).view(np.uint32)


ADVERSARIAL = [float("nan"), float("inf"), -float("inf"), 0.0, -0.0, 0.4, -0.4, 0.5, -0.5, 0.99, -0.99, 1.0, -1.0, 2.5, -2.5,
               3.0, 7.75, -7.75, 80.0, 80.5, 159.0, 159.99, 160.0, 160.5, 161.0, -1.5, 209.5, 210.0, 211.0, 12000.0,
               16383.5, 16384.0, 29999.0, 30000.0, 30000.5, 30001.0, -29999.0, -30000.0, -30000.5, -30001.0, 32767.0, 32768.0,
               -32768.0, 60000.0, -60000.0, 536870911.0, 536870912.0, 536870912.5, 536870913.0, -536870911.0, -536870912.0,
               -536870913.0, 2147483647.0, 2147483648.0, -2147483649.0, 1e12, -1e12, 1e300, -1e300, 5e-324]


def test_mover_rec_equals_mover_on_game_records(L):
    """every record of a random and a ball-tracking rollout, all five movers"""
    e = emu_lib.Emu("breakout")
    e.seed(5)
    e.new_game()
    n = 0
    for t in range(2000):
        e.step(ale_action=[0, 1, 3, 4][(t * 7 + t // 13) % 4], auto_reset=True)
        if t % 7 == 0:
            ref, new = _movers(L, e.record())
            assert np.array_equal(ref, new), (t, ref, new)
            n += int((ref[1:N_MOVERS + 1, 0] < ref[1:N_MOVERS + 1, 2]).sum())
    assert n > 200  # the paddle and a ball were really on the canvas


def test_mover_rec_equals_mover_on_adversarial_records(L):
    """NaN, infinities, +-2^29 and beyond, +-30,000 and beyond, fractional and negative positions, zero and negative sizes,
    0..4 balls (and out-of-range counts), off-canvas balls"""
    e = emu_lib.Emu("breakout")
    W = _words(L)
    base = np.array(e.record(), np.uint32)
    rng = np.random.default_rng(2024)
    vals = np.array(ADVERSARIAL)
    checked = 0

    def check(rec):
        nonlocal checked
        ref, new = _movers(L, rec)
        assert np.array_equal(ref, new), (rec[W["paddle_px"]:W["paddle_px"] + 6].view(np.float64), ref, new)
        checked += 1

    # the paddle: every (x, width) pair of the list, y from a few rows, and the y axis with the width fixed
    for px, pw in itertools.product(vals, vals):
        rec = base.copy()
        _set_f64(rec, W["paddle_px"], px)
        _set_f64(rec, W["paddle_width"], pw)
        _set_f64(rec, W["paddle_py"], [190.0, -1.0, 209.0, float("nan")][checked % 4])
        check(rec)
    for py, pw in itertools.product(vals, [0.0, -3.0, 24.0, 1e9]):
        rec = base.copy()
        _set_f64(rec, W["paddle_px"], 80.0)
        _set_f64(rec, W["paddle_width"], pw)
        _set_f64(rec, W["paddle_py"], py)
        check(rec)
    # the balls: every (x, radius) and (y, radius) pair, with 0..4 balls and counts outside that range
    for (bx, r), nb in itertools.product(itertools.product(vals, vals), [4]):
        rec = base.copy()
        rec[W["n_balls"]] = np.uint32(nb)
        _set_f64(rec, W["ball_radius"], r)
        for b in range(4):
            _set_f64(rec, W["ball"] + 8 * b, bx if b % 2 == 0 else 80.0)
            _set_f64(rec, W["ball"] + 8 * b + 2, 100.0 if b % 2 == 0 else bx)
        check(rec)
    for nb in [-1, 0, 1, 2, 3, 4, 5, 1 << 31]:
        for r in [1.5, 0.0, -2.0, 20000.0, float("nan")]:
            rec = base.copy()
            rec[W["n_balls"]] = np.uint32(nb & 0xFFFFFFFF)
            _set_f64(rec, W["ball_radius"], r)
            for b in range(4):
                _set_f64(rec, W["ball"] + 8 * b, [-10.0, 80.0, 170.0, 5.0][b])
                _set_f64(rec, W["ball"] + 8 * b + 2, [100.0, -5.0, 215.0, 205.0][b])
            check(rec)
    # random mixtures: listed values plus random reals at every scale
    for _ in range(3000):
        rec = base.copy()
        pick = lambda: float(rng.choice(vals)) if rng.random() < 0.5 else float(rng.normal() * 10.0 ** rng.integers(0, 10))
        for w in (W["paddle_px"], W["paddle_py"], W["paddle_width"], W["ball_radius"]):
            _set_f64(rec, w, pick())
        rec[W["n_balls"]] = np.uint32(int(rng.integers(0, 6)))
        for b in range(4):
            _set_f64(rec, W["ball"] + 8 * b, pick())
            _set_f64(rec, W["ball"] + 8 * b + 2, pick())
        check(rec)
    assert checked > 9000


def _accepted_sizes():
    e = emu_lib.Emu("breakout")
    sizes = []
    for w in range(4, 161, 4):                   # the direct kernel needs a width that is a multiple of 4
        for h in list(range(8, 129, 3)) + [84, 105, 210]:
            try:
                info = e.direct_info(w, h)
            except ValueError:
                continue
            if info["ok"] and info["taps"][0] <= 5 and info["taps"][1] <= 4:
                sizes.append((w, h))
    return e, sizes


CACHED = (0, 1, 2, 3, 10, 11)  # the slots the kernel keeps in shared memory: score digits 0..3, lives digits 0..1


def test_cached_digit_patches_never_share_a_pixel(L):
    """at every output size the Breakout direct kernel accepts: the output rectangles of the patches of two different cached
    digit slots (any digits) are disjoint, so the kernel may write their pixels in any order.  A cached slot may share pixels
    with an uncached one only when the uncached one comes later in slot order (lives digits 4.. over the score's low
    digits): those go out one patch at a time after the cached pass, in slot order, as before."""
    e, sizes = _accepted_sizes()
    assert (84, 84) in sizes and len(sizes) > 50
    for w, h in sizes:
        boxes = np.zeros((32 * 10, 4), np.int32)
        ns = L.dc_digit_patch_boxes(w, h, boxes.ctypes.data_as(C.c_void_p))
        assert ns > 0, (w, h)
        boxes = boxes.reshape(32, 10, 4)
        # per slot the union of its digits' rectangles (the score's and the lives' 20 slots are Breakout's)
        occ = np.zeros((20, h, w), bool)
        for s in range(20):
            for d in range(10):
                x0, y0, pw, ph = (int(v) for v in boxes[s, d])
                if pw:
                    occ[s, y0:y0 + ph, x0:x0 + pw] = True
        for s in CACHED:
            assert occ[s].any(), (w, h, s)
            for t in range(20):
                if t == s or not (occ[s] & occ[t]).any():
                    continue
                assert t not in CACHED and t > s, (w, h, s, t)
