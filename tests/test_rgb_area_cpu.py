"""CPU tier: the reference for the colour INTER_AREA layout (TBX_OBS_RGB_AREA) -- the oracle's INTER_AREA resize with 3
interleaved channels (oracle/common.c:tbo_resize_area_u8, cn = 3) of the oracle's RGB frame -- against cv2.resize(rgb, (w, h),
INTER_AREA) itself where cv2 is installed, and always against the committed digests of cv2's outputs (tests/golden/rgb_area_cv2.json,
written by `python tests/test_rgb_area_cpu.py --write-golden` where cv2 is installed); and the rule the RGB tile kernel is built on:
each channel of the result is the single-channel resize of that channel.  tests/test_gpu_rgb_area.py compares the GPU with
rgb_area() below."""
import ctypes as C
import functools
import hashlib
import json
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DIMS = {"breakout": (240, 160), "amidar": (160, 250), "space_invaders": (320, 210)}
# the WarpFrame sizes, uneven and extreme ones, and per game the accepted size with the largest tile-kernel window (8 x 8 taps)
SIZES = [(84, 84), (64, 64), (96, 80), (92, 83), (128, 128), (100, 37)]
WORST_SIZE = {"breakout": (32, 20), "space_invaders": (40, 28), "amidar": (23, 35)}


@functools.lru_cache(maxsize=None)
def source_frames(oracle):
    """(name, game, rgb frame uint8[h][w][3]): seeded noise at each native size, then per game the oracle's frame of a fresh game
    and of a game rolled out with the benchmark's action stream"""
    rng = np.random.default_rng(31)
    out = [("noise_" + g, g, rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)) for g, (w, h) in DIMS.items()]
    for g in DIMS:
        ref = oracle.OracleBatch(g, 1, seeds=[9])
        out.append(("fresh_" + g, g, ref.render("rgb")[0]))
        legal = np.asarray(oracle.LEGAL[g], np.int32)
        for t in range(250):
            ref.step(legal[[oracle.action_index(0xB200, 0, t, len(legal))]], auto_reset=True)
        out.append(("rolled_" + g, g, ref.render("rgb")[0]))
    return out


def sizes(game):
    return SIZES + [WORST_SIZE[game]]


def rgb_area(oracle, rgb, w, h):
    """the oracle's colour INTER_AREA observation of one RGB frame uint8[h][w][3] (or of a batch [n][h][w][3])"""
    if rgb.ndim == 4:
        return np.stack([_resize(oracle, f, 3, w, h) for f in rgb])
    return _resize(oracle, rgb, 3, w, h)


def _resize(oracle, src, cn, w, h):
    sh, sw = src.shape[:2]
    got = np.empty((h, w, cn) if cn > 1 else (h, w), np.uint8)
    src = np.ascontiguousarray(src)
    oracle.lib().tbo_resize_area_u8(src.ctypes.data_as(C.c_void_p), sw, sh, cn, got.ctypes.data_as(C.c_void_p), w, h)
    return got


def test_rgb_area_equals_cv2(oracle_mod):
    try:
        import cv2
    except ImportError:
        cv2 = None
    kat = json.load(open(os.path.join(GOLD, "rgb_area_cv2.json")))
    frames = source_frames(oracle_mod)
    assert [f[0] for f in frames] == list(kat["src_sha256"])
    checked = 0
    for name, game, src in frames:
        assert hashlib.sha256(src.tobytes()).hexdigest() == kat["src_sha256"][name], ("source frame changed: regenerate the digests", name)
        for w, h in sizes(game):
            got = rgb_area(oracle_mod, src, w, h)
            key = "%s_%dx%d" % (name, w, h)
            assert hashlib.sha256(got.tobytes()).hexdigest() == kat["dst_sha256"][key], key
            if cv2 is not None:
                assert np.array_equal(got, cv2.resize(src, (w, h), interpolation=cv2.INTER_AREA)), key
            checked += 1
    assert checked == len(kat["dst_sha256"])


def test_rgb_area_is_the_per_channel_resize(oracle_mod):
    for name, game, src in source_frames(oracle_mod):
        for w, h in sizes(game):
            got = _resize(oracle_mod, src, 3, w, h)
            for c in range(3):
                assert np.array_equal(got[..., c], _resize(oracle_mod, src[..., c], 1, w, h)), (name, w, h, c)


def write_golden():
    """rgb_area_cv2.json: SHA-256 of the source frames above and of cv2's 3-channel INTER_AREA output of each at each of its sizes"""
    import sys
    import cv2
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from oracle import oracle
    out = {"cv2_version": cv2.__version__, "src_sha256": {}, "dst_sha256": {}}
    for name, game, src in source_frames(oracle):
        out["src_sha256"][name] = hashlib.sha256(src.tobytes()).hexdigest()
        for w, h in sizes(game):
            dst = cv2.resize(src, (w, h), interpolation=cv2.INTER_AREA)
            out["dst_sha256"]["%s_%dx%d" % (name, w, h)] = hashlib.sha256(dst.tobytes()).hexdigest()
    json.dump(out, open(os.path.join(GOLD, "rgb_area_cv2.json"), "w"), indent=1)


if __name__ == "__main__":
    import sys
    if sys.argv[1:] == ["--write-golden"]:
        write_golden()
