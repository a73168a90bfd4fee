"""CPU tier: the shared-memory image of the Breakout direct kernel (tbx_direct.h, tbx::build_brk_img), checked on a host build of
the same headers (tests/emu/brk_img_check.cpp).

The kernel copies the image whole into shared memory and reads every table of its per-env path from it, at the offsets of
brk_img_layout.  At every output size the kernel accepts, for the default config and for edited brick configs: each region
equals the table it replaces byte for byte, the regions are 16-byte aligned and do not overlap, and the kernel's shared memory
(image, record stages, per-warp scratch) fits a CTA -- at 84x84 still four CTAs per SM.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

_HERE = os.path.dirname(os.path.abspath(__file__))
REGIONS = ("flags", "dig", "rowcls", "inv", "xdlo", "xdhi", "ydlo", "ydhi", "xcol", "yrow", "bgray", "wordcols", "col0", "dyrows",
           "hsel", "base1", "plan", "hlut", "hstatic", "cls")
SMEM_OPTIN = 227 * 1024          # shared memory a CTA may opt in to on sm_100
SMEM_4_PER_SM = 56320            # (228 KB - 4 x 1 KB reserved) / 4: four CTAs per SM


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """tests/emu/brk_img_check.cpp with the library's host half, built in a temporary directory"""
    so = str(tmp_path_factory.mktemp("brk_img_check") / "libbrk_img_check.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", so,
                           os.path.join(_HERE, "emu", "brk_img_check.cpp"),
                           os.path.join(os.path.dirname(_HERE), "toybox_b200", "csrc", "tbx_host.cpp")])
    lib = C.CDLL(so)
    lib.dc_brk_img.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p]
    return lib


def _image(L, w, h, rows):
    info = np.zeros(27, np.int32)
    r = L.dc_brk_img(w, h, rows, info.ctypes.data_as(C.c_void_p))
    return r, info


def _kernel_smem(info, w):
    """the launcher's dynamic shared memory (tbx_launch_direct): the image, two record stages of 8 envs, 8 warps' H rows and
    mover records"""
    nrows, rw, img_bytes = int(info[2]), int(info[5]), int(info[-1])
    hs = (w + 3) & ~3
    warp_bytes = ((nrows * hs * 4 + 15) & ~15) + 256
    return img_bytes + 2 * rw * 8 * 4 + 8 * warp_bytes


def _sizes():
    for w in range(4, 161, 4):                   # the direct kernel needs a width that is a multiple of 4
        for h in list(range(8, 129, 3)) + [84, 105, 210]:
            yield w, h


@pytest.mark.parametrize("rows", [0, 1, 4, 8])   # 0: the default config (6 rows); else that many brick rows, other colours
def test_image_regions_match_their_tables(L, rows):
    n = 0
    for w, h in _sizes():
        r, info = _image(L, w, h, rows)
        if r == -1:                              # not covered by the direct kernel at this size
            continue
        n += 1
        bad = REGIONS[r - 1] if 0 < r <= len(REGIONS) else r
        assert r == 0, (w, h, rows, "region differs from its table:", bad)
        offs = [int(v) for v in info[6:]]
        assert all(o % 16 == 0 for o in offs), (w, h, rows, offs)
        assert offs == sorted(offs), (w, h, rows, offs)
        assert _kernel_smem(info, w) <= SMEM_OPTIN, (w, h, rows, _kernel_smem(info, w))
    assert n > 50, n


def test_image_at_84x84_keeps_four_ctas_per_sm(L):
    for rows in (0, 8):
        r, info = _image(L, 84, 84, rows)
        assert r == 0 and tuple(info[:2]) == (4, 3), (rows, r, info[:2])
        assert info[4] == 1                      # the cached digit slots' patches are in the image
        assert _kernel_smem(info, 84) <= SMEM_4_PER_SM, (rows, _kernel_smem(info, 84))
