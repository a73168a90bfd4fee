"""ctypes wrapper of tests/emu/libtbx_emu.so -- the TEST-ONLY host build of the engine headers the CUDA
kernels are compiled from (see tests/emu/emu.cpp).  Lets the CPU-only test tier compare the product's
transition / draw-list / resize / JSON code with the oracle without a GPU.  Never imported by the product."""
import ctypes as C
import json
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_LIB = None


def build(force=False):
    so = os.path.join(_HERE, "emu", "libtbx_emu.so")
    src_dir = os.path.join(_ROOT, "toybox_b200", "csrc")
    srcs = [os.path.join(_HERE, "emu", "emu.cpp")] + [os.path.join(src_dir, f) for f in os.listdir(src_dir)
                                                       if f.endswith((".h", ".cpp"))]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", so,
                               os.path.join(_HERE, "emu", "emu.cpp"), os.path.join(src_dir, "tbx_host.cpp")])
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        L.emu_create.restype = C.c_void_p
        L.emu_create.argtypes = [C.c_char_p, C.c_char_p]
        L.emu_last_error.restype = C.c_char_p
        L.emu_record.restype = C.POINTER(C.c_uint32)
        for f in ("emu_state_to_json", "emu_config_to_json", "emu_schema_for_state", "emu_schema_for_config"):
            getattr(L, f).restype = C.c_void_p
        for f in ("emu_destroy", "emu_rec_words", "emu_record", "emu_new_game", "emu_state_to_json", "emu_config_to_json",
                  "emu_n_tables"):
            getattr(L, f).argtypes = [C.c_void_p]
        L.emu_seed.argtypes = [C.c_void_p, C.c_uint32]
        L.emu_step.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.emu_render.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.emu_state_from_json.argtypes = [C.c_void_p, C.c_char_p]
        L.emu_config_from_json.argtypes = [C.c_void_p, C.c_char_p]
        L.emu_schema_for_state.argtypes = [C.c_char_p]
        L.emu_schema_for_config.argtypes = [C.c_char_p]
        L.emu_free_str.argtypes = [C.c_void_p]
        L.emu_action_index.restype = C.c_uint32
        L.emu_action_index.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32]
        _LIB = L
    return _LIB


DIMS = {"breakout": (240, 160), "amidar": (160, 250), "space_invaders": (320, 210)}
MODES = {"rgba": 0, "rgb": 1, "gray": 2, "gray84": 3}


def _take(ptr):
    if not ptr:
        raise ValueError(lib().emu_last_error().decode())
    s = C.string_at(ptr).decode()
    lib().emu_free_str(ptr)
    return s


class Emu:
    def __init__(self, game, cfg_json=None):
        self.game = game
        self.L = lib()
        cfg = json.dumps(cfg_json).encode() if cfg_json is not None else None
        self.h = self.L.emu_create(game.encode(), cfg)
        if not self.h:
            raise ValueError(self.L.emu_last_error().decode())

    def __del__(self):
        if getattr(self, "h", None):
            self.L.emu_destroy(self.h)
            self.h = None

    def seed(self, seed):
        self.L.emu_seed(self.h, seed & 0xFFFFFFFF)

    def new_game(self):
        self.L.emu_new_game(self.h)

    def step(self, ale_action=None, input_mask=None, auto_reset=False):
        out = (C.c_int32 * 4)()
        rc = self.L.emu_step(self.h, -1 if ale_action is None else int(ale_action), -1 if input_mask is None else int(input_mask),
                             int(auto_reset), out)
        if rc != 0:
            raise ValueError("Expected to apply action, but failed: {0}".format(ale_action))
        return out[0], bool(out[1]), out[2], out[3]

    def render(self, mode, out_w=84, out_h=84):
        w, h = DIMS[self.game]
        shape = {"rgba": (h, w, 4), "rgb": (h, w, 3), "gray": (h, w), "gray84": (out_h, out_w)}[mode]
        out = np.empty(shape, np.uint8)
        if self.L.emu_render(self.h, MODES[mode], out_w, out_h, out.ctypes.data_as(C.c_void_p)) != 0:
            raise ValueError(self.L.emu_last_error().decode())
        return out

    def render_fast(self, out_w=84, out_h=84):
        """The fused kernel's INTER_AREA algorithm (base frame + dirty rectangles), emulated on the host."""
        out = np.empty((out_h, out_w), np.uint8)
        self.L.emu_render_fast.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        if self.L.emu_render_fast(self.h, out_w, out_h, out.ctypes.data_as(C.c_void_p)) != 0:
            raise ValueError(self.L.emu_last_error().decode())
        return out

    def render_direct(self, out_w=84, out_h=84):
        """The direct INTER_AREA algorithm (tbx_direct.h) emulated on the host; None when the env is one the kernel hands
        to the general tile kernel."""
        out = np.empty((out_h, out_w), np.uint8)
        self.L.emu_render_direct.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        rc = self.L.emu_render_direct(self.h, out_w, out_h, out.ctypes.data_as(C.c_void_p))
        if rc < 0:
            raise ValueError(self.L.emu_last_error().decode())
        return None if rc else out

    def si_score_strip(self, out_w=84, out_h=84):
        """Space Invaders: the reference frame with the score's pixels taken from the digit-pair table (TbxSiDirect.sc_px), as the
        direct kernel does; None when the table does not exist for this size."""
        out = np.empty((out_h, out_w), np.uint8)
        self.L.emu_si_score_strip.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        rc = self.L.emu_si_score_strip(self.h, out_w, out_h, out.ctypes.data_as(C.c_void_p))
        if rc < 0:
            raise ValueError(self.L.emu_last_error().decode())
        return None if rc else out

    def direct_info(self, out_w=84, out_h=84):
        """The direct INTER_AREA kernel's tables for this config at out_w x out_h, as the library builds them: {"ok"} for
        every game, plus {"nrows", "n_cls"} for Breakout and {"n_sets", "sc_ok"} for Space Invaders.  ok == 0: the tile
        kernel renders every env of that size; n_sets == 0: no sprite patch tables; sc_ok == 0: no score strip.  "taps" is
        the resize plan's (taps per output column, taps per output row); wrapped observations take at most (5, 4)."""
        out = (C.c_int32 * 5)()
        self.L.emu_direct_info.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        if self.L.emu_direct_info(self.h, out_w, out_h, out) != 0:
            raise ValueError(self.L.emu_last_error().decode())
        info = {"ok": out[0], "taps": (out[3], out[4])}
        if self.game == "breakout":
            info.update(nrows=out[1], n_cls=out[2])
        elif self.game == "space_invaders":
            info.update(n_sets=out[1], sc_ok=out[2])
        return info

    def state_json(self):
        return json.loads(_take(self.L.emu_state_to_json(self.h)))

    def write_state_json(self, js):
        if self.L.emu_state_from_json(self.h, json.dumps(js).encode()) != 0:
            raise ValueError(self.L.emu_last_error().decode())

    def config_json(self):
        return json.loads(_take(self.L.emu_config_to_json(self.h)))

    def write_config_json(self, js):
        if self.L.emu_config_from_json(self.h, json.dumps(js).encode()) != 0:
            raise ValueError(self.L.emu_last_error().decode())

    def record(self):
        n = self.L.emu_rec_words(self.h)
        return np.ctypeslib.as_array(self.L.emu_record(self.h), shape=(n,)).copy()

    def n_tables(self):
        return self.L.emu_n_tables(self.h)


def schema_for_state(game):
    return json.loads(_take(lib().emu_schema_for_state(game.encode())))


def schema_for_config(game):
    return json.loads(_take(lib().emu_schema_for_config(game.encode())))
