"""Regenerates the golden fixtures under tests/golden/ (run in the build container, where /root/reference and
cv2 exist; the fixtures travel, the reference does not).

  *_config_default.json, *_state_default.json   the reference's own default fixtures
                                                (toybox/interventions/defaults/), the only complete states it pins
  rng_kat.json                                  xoroshiro128+ known answers derived from those fixtures (SURVEY App. A)
  area_golden.npz                               cv2.resize(..., INTER_AREA) outputs for the three native frame sizes
  reference_py/                                 byte-identical snapshot of the pure-Python reference files its own unit tests
                                                need (toybox/interventions/*.py + defaults, toybox/envs/atari/constants.py,
                                                test/interventions/*.py), so that tests/test_reference_suite.py can run them
                                                on the GPU box -- where /root/reference does not exist -- against the CUDA path
                                                (toybox_b200.ctoybox.Toybox).  Test fixtures, never imported by the product.
"""
import json
import os
import shutil

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference/toybox/interventions/defaults"


def snapshot_reference_py():
    root = "/root/reference"
    dst = os.path.join(HERE, "reference_py")
    shutil.rmtree(dst, ignore_errors=True)
    files = ["toybox/__init__.py", "toybox/envs/atari/constants.py", "test/__init__.py", "test/interventions/__init__.py"]
    for d in ("toybox/interventions", "test/interventions"):
        files += [os.path.join(d, f) for f in sorted(os.listdir(os.path.join(root, d))) if f.endswith(".py")]
    files += [os.path.join("toybox/interventions/defaults", f) for f in sorted(os.listdir(os.path.join(root, "toybox/interventions/defaults")))]
    for f in files:
        src = os.path.join(root, f)
        os.makedirs(os.path.dirname(os.path.join(dst, f)), exist_ok=True)
        if os.path.exists(src):
            shutil.copyfile(src, os.path.join(dst, f))
        else:
            open(os.path.join(dst, f), "w").close()          # package marker the reference does not ship
    with open(os.path.join(dst, "README"), "w") as fh:
        fh.write("Byte-identical copies of files of /root/reference (toybox-rs/Toybox), made by tests/golden/make_golden.py.\n"
                 "Test fixtures only: tests/test_reference_suite.py runs the reference's own unit tests from here where the\n"
                 "reference tree is absent (the GPU box).  Nothing under toybox_b200/ imports them.\n")


def main():
    snapshot_reference_py()
    for g in ("breakout", "amidar", "space_invaders"):
        for kind in ("config", "state"):
            shutil.copyfile(os.path.join(REF, "%s_%s_default.json" % (g, kind)), os.path.join(HERE, "%s_%s_default.json" % (g, kind)))
    kat = {
        "seed_state": [1817879012901901412, 10917585336602961851],
        "outputs": [12735464349504863263, 9270897318777222480, 1639874325333928636, 2870494946185607049,
                    5980051464858656592, 16111260417487562734],
        "state_after_6": [8317881511975408900, 11692541923059621836],
        "breakout_child_draws": [4510369271519535685, 9330771300662569460],
        "breakout_child_born": [1639874325333928636, 2870494946185607049],
        "si_config_before": [14726119713774332226, 5397374105704621022],
    }
    json.dump(kat, open(os.path.join(HERE, "rng_kat.json"), "w"), indent=1)
    import cv2
    rng = np.random.default_rng(20261017)
    out = {"cv2_version": np.array(cv2.__version__)}
    for name, (w, h) in {"breakout": (240, 160), "amidar": (160, 250), "space_invaders": (320, 210)}.items():
        img = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
        blocky = np.kron(rng.integers(0, 256, size=(h // 10, w // 10), dtype=np.uint8), np.ones((10, 10), np.uint8))
        out[name + "_src_noise"] = img
        out[name + "_dst_noise"] = cv2.resize(img, (84, 84), interpolation=cv2.INTER_AREA)
        out[name + "_src_blocky"] = blocky
        out[name + "_dst_blocky"] = cv2.resize(blocky, (84, 84), interpolation=cv2.INTER_AREA)
        out[name + "_dst_noise_100x60"] = cv2.resize(img, (100, 60), interpolation=cv2.INTER_AREA)
    np.savez_compressed(os.path.join(HERE, "area_golden.npz"), **out)
    area_cv2_seed5()


def area_cv2_seed5():
    """area_cv2_seed5.json: SHA-256 of the noise frames of tests/test_oracle_golden.py::test_area_resize_equals_live_cv2
    (default_rng(5), 5 per game) and of their cv2 INTER_AREA 84x84 outputs."""
    import hashlib
    import cv2
    rng = np.random.default_rng(5)
    out = {"cv2_version": cv2.__version__, "src_sha256": [], "dst_sha256": []}
    for (w, h) in ((240, 160), (160, 250), (320, 210)):
        for _ in range(5):
            src = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
            out["src_sha256"].append(hashlib.sha256(src.tobytes()).hexdigest())
            out["dst_sha256"].append(hashlib.sha256(cv2.resize(src, (84, 84), interpolation=cv2.INTER_AREA).tobytes()).hexdigest())
    json.dump(out, open(os.path.join(HERE, "area_cv2_seed5.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
