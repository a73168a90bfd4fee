"""BatchedToybox: N device-resident environments of one game behind the method surface of
`ctoybox.Toybox` (reference call sites: toybox/envs/atari/base.py:57-167, toybox/interventions/base.py:387-408),
each method taken to batch size N.  PyTorch supplies device memory and streams; all simulation and
rendering happens in libtoybox_b200.so (hand-written sm_100a kernels)."""
import ctypes as C
import json

import numpy as np
import torch

from . import _lib
from . import snapshot as _snap

GAMES = ("breakout", "amidar", "space_invaders")
OBS_MODES = {"rgba": 0, "rgb": 1, "gray": 2, "gray_area": 3, "rgb_area": 4}


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class BatchedToybox:
    """`n_envs` independent environments of `game` on one CUDA device.

    obs: 'rgba' uint8[N,H,W,4] | 'rgb' uint8[N,H,W,3] | 'gray' uint8[N,H,W,1] | 'gray84' uint8[N,84,84,1]
         (= cv2.INTER_AREA of the grayscale frame, baselines WarpFrame) | ('gray_area', out_w, out_h) | 'rgb84' uint8[N,84,84,3]
         (= cv2.INTER_AREA of the RGB frame, WarpFrame(grayscale=False)) | ('rgb_area', out_w, out_h).
    """

    def __init__(self, game, n_envs, device=None, obs="gray84", config=None, seeds=None):
        if game not in GAMES:
            raise ValueError("unknown game %r (have %s)" % (game, ", ".join(GAMES)))
        if not torch.cuda.is_available():
            raise _lib.ToyboxError("toybox_b200 needs a CUDA device (sm_100a); there is no CPU path")
        self.L = _lib.lib()
        self.game_name = game
        self.n_envs = int(n_envs)
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else torch.device(device).index or 0)
        handle = C.c_void_p()
        cfg = json.dumps(config).encode() if config is not None else None
        _lib.check(self.L.tbx_pool_create(game.encode(), self.n_envs, self.device.index, cfg, C.byref(handle)))
        self._h = handle
        self.width = self.L.tbx_frame_width(self._h)
        self.height = self.L.tbx_frame_height(self._h)
        legal = (C.c_int32 * 18)()
        n = self.L.tbx_legal_actions(self._h, legal, 18)
        self._legal = [int(legal[i]) for i in range(n)]
        self.set_obs(obs)
        dev = self.device
        self.reward = torch.zeros(self.n_envs, dtype=torch.int32, device=dev)
        self.done = torch.zeros(self.n_envs, dtype=torch.uint8, device=dev)
        self.score = torch.zeros(self.n_envs, dtype=torch.int32, device=dev)
        self.lives = torch.zeros(self.n_envs, dtype=torch.int32, device=dev)
        self._obs = None
        if seeds is not None:
            self.set_seed(seeds)
            self.new_game()

    # ------------------------------------------------------------------ life cycle
    def close(self):
        if getattr(self, "_h", None):
            self.L.tbx_pool_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ------------------------------------------------------------------ geometry / actions
    def set_obs(self, obs):
        if isinstance(obs, (tuple, list)):
            mode, ow, oh = obs
        elif obs in ("gray84", "rgb84"):
            mode, ow, oh = obs[:-2] + "_area", 84, 84
        else:
            mode, ow, oh = obs, 0, 0
        if mode not in OBS_MODES:
            raise ValueError("unknown obs layout %r" % (obs,))
        nbytes = self.L.tbx_obs_bytes(self._h, OBS_MODES[mode], ow, oh)
        if nbytes == 0:
            raise ValueError("unsupported observation size %r for %s" % (obs, self.game_name))
        self._mode, self._ow, self._oh, self._obs_bytes = OBS_MODES[mode], ow, oh, nbytes
        H, W = self.height, self.width
        self.obs_shape = {0: (H, W, 4), 1: (H, W, 3), 2: (H, W, 1), 3: (oh, ow, 1), 4: (oh, ow, 3)}[self._mode]
        self._obs = None

    def get_width(self):
        return self.width

    def get_height(self):
        return self.height

    def get_legal_action_set(self):
        return list(self._legal)

    # ------------------------------------------------------------------ seeding / reset
    def set_seed(self, seeds, env_ids=None):
        """Toybox.set_seed per env: `seeds` is an int (env i gets seed+i) or an array of n u32."""
        if np.isscalar(seeds):
            n = self.n_envs if env_ids is None else len(env_ids)
            seeds = (int(seeds) + np.arange(n, dtype=np.int64)) & 0xFFFFFFFF
        seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
        ids = None if env_ids is None else np.ascontiguousarray(env_ids, dtype=np.int32)
        torch.cuda.synchronize(self.device)
        _lib.check(self.L.tbx_seed(self._h, seeds.ctypes.data_as(C.c_void_p), None if ids is None else ids.ctypes.data_as(C.c_void_p),
                                   len(seeds)))

    def new_game(self, mask=None):
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self.L.tbx_new_game(self._h, _ptr(mask), _stream(self.device)))

    # ------------------------------------------------------------------ step / render
    def _actions(self, actions, dtype):
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(np.asarray(actions), dtype=dtype)
        a = actions.to(device=self.device, dtype=dtype, non_blocking=True).contiguous()
        if a.numel() != self.n_envs:
            raise ValueError("expected %d actions, got %d" % (self.n_envs, a.numel()))
        return a

    def apply_ale_action(self, actions, auto_reset=False):
        """Toybox.apply_ale_action for every env; fills self.reward/done/score/lives (device tensors)."""
        a = self._actions(actions, torch.int32)
        _lib.check(self.L.tbx_step(self._h, _ptr(a), int(auto_reset), _ptr(self.reward), _ptr(self.done), _ptr(self.score),
                                   _ptr(self.lives), _stream(self.device)))

    def apply_action(self, inputs, auto_reset=False):
        """Toybox.apply_action(Input) for every env; `inputs` are Input bitmasks (see Input.mask())."""
        a = self._actions(inputs, torch.uint8)
        _lib.check(self.L.tbx_step_inputs(self._h, _ptr(a), int(auto_reset), _ptr(self.reward), _ptr(self.done), _ptr(self.score),
                                          _ptr(self.lives), _stream(self.device)))

    def step_random(self, seed, t, env0=0, auto_reset=True):
        """apply_ale_action with the benchmark's reproducible uniform-over-legal action stream generated inside the step
        kernel (one launch; same states as fill_random_actions + apply_ale_action)."""
        _lib.check(self.L.tbx_step_random(self._h, int(seed), int(env0), int(t), int(auto_reset), _ptr(self.reward), _ptr(self.done),
                                          _ptr(self.score), _ptr(self.lives), _stream(self.device)))

    def check(self):
        """Synchronise and raise ValueError if any env was handed an invalid ALE action id."""
        _lib.check(self.L.tbx_check(self._h, _stream(self.device)))

    def render(self, out=None, obs=None):
        """Toybox.get_state() for every env, written straight into a torch tensor uint8[N, *obs_shape]."""
        if obs is not None:
            saved = (self._mode, self._ow, self._oh, self._obs_bytes, self.obs_shape)
            self.set_obs(obs)
        try:
            if out is None:
                if self._obs is None or obs is not None:
                    out = torch.empty((self.n_envs,) + self.obs_shape, dtype=torch.uint8, device=self.device)
                    if obs is None:
                        self._obs = out
                else:
                    out = self._obs
            if out.numel() != self.n_envs * self._obs_bytes or out.dtype != torch.uint8 or not out.is_contiguous():
                raise ValueError("out must be a contiguous uint8 tensor of %d bytes" % (self.n_envs * self._obs_bytes))
            _lib.check(self.L.tbx_render(self._h, _ptr(out), self._mode, self._ow, self._oh, _stream(self.device)))
        finally:
            if obs is not None:
                self._mode, self._ow, self._oh, self._obs_bytes, self.obs_shape = saved
        return out

    get_state = render

    def get_rgb_frame(self):
        return self.render(obs="rgb")

    def step(self, actions, auto_reset=True, render=True):
        """One batched env.step (toybox/envs/atari/base.py:115-149): returns (obs, reward, done, info tensors)."""
        self.apply_ale_action(actions, auto_reset=auto_reset)
        obs = self.render() if render else None
        return obs, self.reward, self.done.bool(), {"lives": self.lives, "score": self.score}

    def step_host(self, actions, obs_out=None, auto_reset=True):
        """The same step for host-resident callers: numpy/pinned-tensor actions in, host buffers out."""
        a = np.ascontiguousarray(actions.numpy() if torch.is_tensor(actions) else actions, dtype=np.int32)
        n = self.n_envs
        if not hasattr(self, "_h_out"):
            self._h_out = [torch.empty(n, dtype=torch.int32).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory(),
                           torch.empty(n, dtype=torch.int32).pin_memory(), torch.empty(n, dtype=torch.int32).pin_memory()]
        if obs_out is None:
            key = (self._mode, self._ow, self._oh)
            if getattr(self, "_h_obs_key", None) != key:
                self._h_obs = torch.empty((n,) + self.obs_shape, dtype=torch.uint8).pin_memory()
                self._h_obs_key = key
            obs_out = self._h_obs
        r, d, s, l = self._h_out
        _lib.check(self.L.tbx_step_host(self._h, a.ctypes.data_as(C.c_void_p), int(auto_reset), self._mode, self._ow, self._oh,
                                        C.c_void_p(obs_out.data_ptr()), C.c_void_p(r.data_ptr()), C.c_void_p(d.data_ptr()),
                                        C.c_void_p(s.data_ptr()), C.c_void_p(l.data_ptr())))
        return obs_out, r, d, {"score": s, "lives": l}

    def fill_random_actions(self, out, seed, t, env0=0):
        """The benchmark's reproducible uniform-over-legal action stream (SURVEY 8d), generated on the device.  `t` is the
        frame index: a python int, or a one-element int64 device tensor read when the kernel runs (CUDA-graph replays)."""
        if torch.is_tensor(t):
            _lib.check(self.L.tbx_fill_actions_at(self._h, _ptr(out), int(seed), int(env0), _ptr(t), _stream(self.device)))
        else:
            _lib.check(self.L.tbx_fill_actions(self._h, _ptr(out), int(seed), int(env0), int(t), _stream(self.device)))
        return out

    def fill_policy_actions(self, out, policy, t):
        """Benchmark utility: scripted actions from the envs' own state (policy 1: Breakout ball tracking)."""
        _lib.check(self.L.tbx_fill_actions_policy(self._h, _ptr(out), int(policy), int(t), _stream(self.device)))
        return out

    # ------------------------------------------------------------------ scalars
    def _scalars(self):
        score = torch.empty(self.n_envs, dtype=torch.int32, device=self.device)
        lives = torch.empty_like(score)
        level = torch.empty_like(score)
        _lib.check(self.L.tbx_read_scalars(self._h, _ptr(score), _ptr(lives), _ptr(level), _stream(self.device)))
        return score, lives, level

    def get_score(self):
        return self._scalars()[0]

    def get_lives(self):
        return self._scalars()[1]

    def get_level(self):
        return self._scalars()[2]

    def game_over(self):
        return self._scalars()[1] <= 0

    def episode_stats(self, reset=False):
        """[episodes, sum of returns, sum of lengths, max return] since the counters were last reset."""
        out = (C.c_int64 * 4)()
        _lib.check(self.L.tbx_stats_read(self._h, out, int(reset), _stream(self.device)))
        return [int(v) for v in out]

    def episode_stats_into(self, out):
        """The same four counters copied into `out` (int64[4] on the pool's device) in stream order, without a host
        synchronisation -- the form a collective inside a timed region consumes."""
        if out.dtype != torch.int64 or out.numel() != 4 or out.device != self.device:
            raise ValueError("out must be int64[4] on the pool's device")
        _lib.check(self.L.tbx_stats_read_device(self._h, _ptr(out), _stream(self.device)))
        return out

    # ------------------------------------------------------------------ vectorised properties (no JSON round trip)
    def property_info(self, path):
        """(word, kind, bit) of a scalar of the state schema; kind: 0 int32, 1 float64, 2 bool, 3 bit, 4 Option<i32>."""
        w, k, b = C.c_int(), C.c_int(), C.c_int()
        _lib.check(self.L.tbx_field_lookup(self.game_name.encode(), path.encode(), C.byref(w), C.byref(k), C.byref(b)))
        return w.value, k.value, b.value

    def get_property(self, path):
        """`get_property(path)` of toybox/interventions/core.py:285-304 for EVERY env: a device tensor [N] (float64 for the
        f64 fields, bool for booleans, int32 otherwise; Option<i32> None reads as INT32_MIN)."""
        _, kind, _ = self.property_info(path)
        out = torch.empty(self.n_envs, dtype=torch.float64 if kind == 1 else torch.int32, device=self.device)
        _lib.check(self.L.tbx_field_get(self._h, path.encode(), _ptr(out), _stream(self.device)))
        return out.bool() if kind in (2, 3) else out

    def set_property(self, path, values, mask=None):
        """Write one scalar of the state schema for every env (or the envs flagged in `mask`): `values` is a python scalar
        or a tensor/array of N values; None writes an Option<i32> None."""
        _, kind, _ = self.property_info(path)
        dt = torch.float64 if kind == 1 else torch.int32
        if values is None:
            if kind != 4:
                raise ValueError("%s is not an Option field" % path)
            values = -2 ** 31
        if torch.is_tensor(values):
            v = values.to(device=self.device, dtype=dt).contiguous()
        elif np.ndim(values) == 0:
            v = torch.full((self.n_envs,), values, dtype=dt, device=self.device)
        else:
            v = torch.as_tensor(np.ascontiguousarray(values), device=self.device).to(dt).contiguous()
        if v.numel() != self.n_envs:
            raise ValueError("expected %d values" % self.n_envs)
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
            if m.numel() != self.n_envs:
                raise ValueError("expected a mask of %d entries" % self.n_envs)
        _lib.check(self.L.tbx_field_set(self._h, path.encode(), _ptr(v), _ptr(m), _stream(self.device)))

    # ------------------------------------------------------------------ state snapshots (no JSON, no host synchronisation)
    def save_state(self, env_ids=None):
        """A StateSnapshot of the listed envs (all by default; ids may repeat): column j holds env env_ids[j].  Enqueued on the
        current stream.  Ids: a host sequence (checked here) or an int32 device tensor (checked on the device, see check())."""
        ids = _snap.id_tensor(env_ids, self.n_envs, self.device, "env id")
        k = self.n_envs if ids is None else ids.numel()
        data = torch.empty((self.L.tbx_state_rows(self._h), k), dtype=torch.int32, device=self.device)
        _lib.check(self.L.tbx_state_save(self._h, _ptr(ids), k, _ptr(data), _stream(self.device)))
        return _snap.StateSnapshot(data, _snap.tables_blob(self.L.tbx_state_tables, self._h))

    def load_state(self, snap, env_ids=None, columns=None):
        """Env env_ids[j] <- column columns[j] of `snap` (defaults: envs 0.., columns 0..); a loaded env continues exactly as the
        saved one would have.  An env listed twice receives the last listed column.  Snapshots of another pool, config or
        GPU of the same game load too (a snapshot on another device is copied here first)."""
        if getattr(snap, "wrapped", False):
            raise ValueError("this snapshot holds wrapper state: load it into a DeepmindToybox")
        data, ids, cols, n = _snap.load_args(snap, self.device, self.n_envs, env_ids, columns)
        _lib.check(self.L.tbx_state_load(self._h, _ptr(data), data.shape[1], _ptr(cols), _ptr(ids), n, snap.tables, len(snap.tables),
                                         _stream(self.device)))

    def fork(self, src_ids, dst_ids=None):
        """Copy the state of env src_ids[j] into env dst_ids[j] (every env by default); one source may feed every destination."""
        snap = self.save_state(src_ids)
        dst = _snap.id_tensor(dst_ids, self.n_envs, self.device, "env id")
        self.load_state(snap, dst, _snap.fork_columns(snap.k, self.n_envs if dst is None else dst.numel(), self.device))

    # ------------------------------------------------------------------ JSON (interventions)
    def to_state_json_text(self, env_ids=None):
        """Toybox.to_state_json() of the listed envs as JSON TEXT (bytes), one document per env: the batched export without
        the Python object trees (decode only the documents you edit)."""
        ids = np.arange(self.n_envs, dtype=np.int32) if env_ids is None else np.ascontiguousarray(env_ids, dtype=np.int32)
        out = (C.c_void_p * len(ids))()
        torch.cuda.synchronize(self.device)
        _lib.check(self.L.tbx_state_to_json(self._h, ids.ctypes.data_as(C.c_void_p), len(ids), out))
        docs = []
        for p in out:
            docs.append(C.string_at(p))
            self.L.tbx_free_str(p)
        return docs

    def to_state_json(self, env_ids=None):
        return [json.loads(d) for d in self.to_state_json_text(env_ids)]

    state_to_json = to_state_json

    def write_state_json(self, states, env_ids=None):
        """Toybox.write_state_json for the listed envs; `states` holds dicts or JSON text (str / bytes), one per env."""
        ids = np.arange(self.n_envs, dtype=np.int32) if env_ids is None else np.ascontiguousarray(env_ids, dtype=np.int32)
        if len(states) != len(ids):
            raise ValueError("one state per env id expected")
        docs = [s if isinstance(s, bytes) else s.encode() if isinstance(s, str) else json.dumps(s).encode() for s in states]
        arr = (C.c_char_p * len(ids))(*docs)
        torch.cuda.synchronize(self.device)
        _lib.check(self.L.tbx_state_from_json(self._h, ids.ctypes.data_as(C.c_void_p), len(ids), arr))

    def config_to_json(self):
        out = C.c_void_p()
        _lib.check(self.L.tbx_config_to_json(self._h, C.byref(out)))
        return json.loads(_lib.take_str(out))

    def write_config_json(self, config):
        torch.cuda.synchronize(self.device)
        _lib.check(self.L.tbx_config_from_json(self._h, json.dumps(config).encode()))

    def schema_for_state(self):
        return schema_for_state(self.game_name)

    def schema_for_config(self):
        return schema_for_config(self.game_name)

    def query_state_json(self, query, args="null", env_id=0):
        out = C.c_void_p()
        torch.cuda.synchronize(self.device)
        _lib.check(self.L.tbx_query_json(self._h, int(env_id), query.encode(), json.dumps(args).encode() if not isinstance(args, str)
                                         else args.encode(), C.byref(out)))
        return json.loads(_lib.take_str(out))


def schema_for_state(game):
    out = C.c_void_p()
    _lib.check(_lib.lib().tbx_schema_for_state(game.encode(), C.byref(out)))
    return json.loads(_lib.take_str(out))


def schema_for_config(game):
    out = C.c_void_p()
    _lib.check(_lib.lib().tbx_schema_for_config(game.encode(), C.byref(out)))
    return json.loads(_lib.take_str(out))
