"""The callers either side of the hot path (SURVEY 8(f1), 8(f2)), at batch size N on one GPU.

`DeepmindToybox` is the reference's wrapper stack
    make_atari:    MaxAndSkipEnv(NoopResetEnv(env, 30), 4)             baselines/baselines/common/atari_wrappers.py:323-333
    wrap_deepmind: FrameStack(ClipRewardEnv(WarpFrame(FireResetEnv(EpisodicLifeEnv(env)))), 4)          :345-360
fused into two kernel launches per agent step (tbx_wrap_step: csrc/tbx_wrap.cuh + the dual mode of
csrc/tbx_render_area.cuh).  `ToyboxVecEnv` gives it the VecEnv surface baselines' trainers consume
(baselines/baselines/common/vec_env/__init__.py:26-131: reset / step_async / step_wait / step / close, num_envs,
observation_space, action_space; auto-reset and `infos[i]['episode']` as vec_env/subproc_vec_env.py:11-15 +
bench/monitor.py:58-76 provide them).
"""
import ctypes as C
import json
import os
import time

import numpy as np
import torch

from . import _lib
from . import snapshot as _snap
from .pool import OBS_MODES, BatchedToybox, _ptr, _stream


class DeepmindToybox:
    """N wrapped envs.  step(actions) takes gym action INDICES (0..len(legal)-1, envs/atari/base.py:126) as an int32
    tensor on the pool's device and returns (obs, reward, done, info):
      obs    uint8[N, k, out_h, out_w] (uint8[N, k, out_h, out_w, 3] when grayscale=False): a RING of the last k
             observations per env -- the newest is obs[:, self.slot], FrameStack order (oldest first) is slots
             (self.slot + 1 .. self.slot + k) % k; `stacked()` returns that order as the reference's
             uint8[N, out_h, out_w, k] (uint8[N, out_h, out_w, 3k] in colour) (a copy);
      reward int32[N] (sign of the summed reward when clip_rewards), done uint8[N] (game over, a lost life when
      episode_life, or the time limit), info = {'lives', 'score', 'real_done', 'truncated', 'ep_return', 'ep_length'}
      tensors (values before the reset of a finished env; truncated: the time limit ended the episode before its game
      was over, all zero without a limit; ep_return / ep_length: Monitor's record where real_done or truncated).
    A finished env is reset inside the same call and `obs` then holds its reset observation (VecEnv semantics)."""

    def __init__(self, game, n_envs, device=None, seeds=None, config=None, frame_skip=4, noop_max=30, episode_life=True,
                 fire_reset=True, clip_rewards=True, frame_stack=4, size=(84, 84), noop_seed=0, env0=0, stack_reset="fill",
                 grayscale=True, repeat_action_probability=0.0, sticky_seed=None, max_episode_steps=None):
        """stack_reset: what a reset observation does to the other k-1 ring slots -- "fill" (FrameStack.reset,
        atari_wrappers.py:262-266: wrap_deepmind(frame_stack=True), the deepq path) or "zero" (VecFrameStack,
        vec_env/vec_frame_stack.py:17-30: make_vec_env + VecFrameStack, the ppo2 / a2c path of run.py:123-125).
        grayscale: WarpFrame's argument (atari_wrappers.py:230-244); False gives colour observations, the INTER_AREA
        down-sample of the pixel-wise max of the last two RGB frames.
        repeat_action_probability: sticky actions (Machado et al. 2018; ALE v5 uses 0.25) on every game frame the stack
        runs, reset-chain frames included: with this probability a frame repeats the ALE id of the env's previous frame
        instead of applying the requested one.  The draws are counter-based, keyed by (sticky_seed, env0 + i, frame);
        sticky_seed defaults to noop_seed.
        max_episode_steps: gym's TimeLimit inside make_atari (baselines' make_atari(env_id, max_episode_steps); ALE v5's
        108,000 frames are 27,000 at frame_skip 4), counting Monitor's episode length.  An env at the limit reports done
        and takes the full reset chain; info['truncated'] flags it where its game is not over."""
        if stack_reset not in ("fill", "zero"):
            raise ValueError("stack_reset is 'fill' (FrameStack) or 'zero' (VecFrameStack)")
        self.pool = BatchedToybox(game, n_envs, device=device, obs=("gray_area", size[0], size[1]), config=config, seeds=seeds)
        self.L = self.pool.L
        self.n_envs, self.device = self.pool.n_envs, self.pool.device
        self.k, self.out_w, self.out_h = int(frame_stack), int(size[0]), int(size[1])
        self.grayscale = bool(grayscale)
        self.frame_shape = (self.out_h, self.out_w) if self.grayscale else (self.out_h, self.out_w, 3)
        h = C.c_void_p()
        _lib.check(self.L.tbx_wrap_create(self.pool._h, int(frame_skip), int(noop_max), int(bool(episode_life)), int(bool(fire_reset)),
                                          int(bool(clip_rewards)), self.k, self.out_w, self.out_h, int(noop_seed), int(env0), C.byref(h)))
        self._w = h
        _lib.check(self.L.tbx_wrap_set_stack_mode(self._w, 1 if stack_reset == "zero" else 0))
        if not self.grayscale:
            _lib.check(self.L.tbx_wrap_set_obs_mode(self._w, OBS_MODES["rgb_area"]))
        self.repeat_action_probability = float(repeat_action_probability)
        self.max_episode_steps = None if max_episode_steps is None else int(max_episode_steps)
        if self.repeat_action_probability != 0.0:
            seed = noop_seed if sticky_seed is None else sticky_seed
            _lib.check(self.L.tbx_wrap_set_sticky_actions(self._w, self.repeat_action_probability, int(seed)))
        n, dev = self.n_envs, self.device
        self.truncated = torch.zeros(n, dtype=torch.uint8, device=dev)
        _lib.check(self.L.tbx_wrap_set_time_limit(self._w, self.max_episode_steps or 0, _ptr(self.truncated)))
        # Monitor's episode record (bench/monitor.py:58-76) of the episode that ended in the last agent step, where real_done or truncated
        self.ep_return = torch.zeros(n_envs, dtype=torch.int32, device=self.device)
        self.ep_length = torch.zeros(n_envs, dtype=torch.int32, device=self.device)
        _lib.check(self.L.tbx_wrap_set_episode_outputs(self._w, _ptr(self.ep_return), _ptr(self.ep_length)))
        self.obs = torch.zeros((n, self.k) + self.frame_shape, dtype=torch.uint8, device=dev)
        self.reward = torch.zeros(n, dtype=torch.int32, device=dev)
        self.done = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.real_done = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.score = torch.zeros(n, dtype=torch.int32, device=dev)
        self.lives = torch.zeros(n, dtype=torch.int32, device=dev)
        self.slot = 0
        self.n_actions = len(self.pool.get_legal_action_set())

    def close(self):
        if getattr(self, "_w", None):
            self.L.tbx_wrap_destroy(self._w)
            self._w = None
        self.pool.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _call(self, actions, render=True):
        slot = C.c_int(0)
        _lib.check(self.L.tbx_wrap_step(self._w, _ptr(actions), _ptr(self.obs) if render else None, _ptr(self.reward), _ptr(self.done),
                                        _ptr(self.real_done), _ptr(self.score), _ptr(self.lives), C.byref(slot), _stream(self.device)))
        self.slot = slot.value

    def reset(self):
        """env.reset() of every wrapped env (a new game only where the last one is over, as EpisodicLifeEnv.reset)."""
        self._call(None)
        return self.obs

    def step(self, actions, render=True):
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(np.ascontiguousarray(actions, dtype=np.int32), device=self.device)
        if actions.dtype != torch.int32 or actions.device != self.device or not actions.is_contiguous() or actions.numel() != self.n_envs:
            actions = actions.to(device=self.device, dtype=torch.int32).contiguous()
            if actions.numel() != self.n_envs:
                raise ValueError("expected %d actions" % self.n_envs)
        self._call(actions, render)
        return self.obs, self.reward, self.done, {"lives": self.lives, "score": self.score, "real_done": self.real_done,
                                                    "truncated": self.truncated, "ep_return": self.ep_return, "ep_length": self.ep_length}

    def check(self):
        self.pool.check()

    # ------------------------------------------------------------------ state snapshots
    def save_state(self, env_ids=None):
        """A StateSnapshot of the listed wrapped envs: records, wrapper state (EpisodicLife, no-op reset counter, Monitor
        accumulators, and with sticky actions the remembered ALE id and frame counter) and observation rings.  Ids as
        BatchedToybox.save_state."""
        ids = _snap.id_tensor(env_ids, self.n_envs, self.device, "env id")
        k = self.n_envs if ids is None else ids.numel()
        data = torch.empty((self.L.tbx_wrap_state_rows(self._w), k), dtype=torch.int32, device=self.device)
        _lib.check(self.L.tbx_wrap_state_save(self._w, _ptr(ids), k, _ptr(data), _stream(self.device)))
        # device ids are checked by the kernel; clamped here only so that the gather cannot fault (skipped entries are reported)
        obs = self.obs.clone() if ids is None else self.obs.index_select(0, ids.long().clamp(0, self.n_envs - 1))
        return _snap.StateSnapshot(data, _snap.tables_blob(self.L.tbx_wrap_state_tables, self._w), wrapped=True, obs=obs, slot=self.slot)

    def load_state(self, snap, env_ids=None, columns=None):
        """Env env_ids[j] <- column columns[j] of a wrapped snapshot, as BatchedToybox.load_state.  Ring rows are rotated so that
        the saved newest frame lands on self.slot: stacked() then equals its value at the moment of the save.  Synchronises
        (the ring copy selects the entries the kernel applied)."""
        if not getattr(snap, "wrapped", False) or tuple(snap.obs.shape[1:]) != tuple(self.obs.shape[1:]):
            raise ValueError("expected a snapshot of wrapped envs with %d x %d x %d observation rings of %d channel%s%s"
                             % (self.k, self.out_h, self.out_w, self.channels, "" if self.channels == 1 else "s", _got_rings(snap)))
        data, ids, cols, n = _snap.load_args(snap, self.device, self.n_envs, env_ids, columns)
        _lib.check(self.L.tbx_wrap_state_load(self._w, _ptr(data), data.shape[1], _ptr(cols), _ptr(ids), n, snap.tables, len(snap.tables),
                                              _stream(self.device)))
        obs = snap.obs if snap.obs.device == self.device else snap.obs.to(self.device)
        shift = (self.slot - snap.slot) % self.k
        if shift:
            obs = torch.roll(obs, shifts=shift, dims=1)
        if ids is None and cols is None:      # env j <- column j: every entry applies unless check() reports skipped ones
            self.obs[:n].copy_(obs[:n])
            return
        # the entries the kernel applied: in range, table index below the blob's count, and the last one for each env
        dev, k = self.device, snap.k
        ids = torch.arange(n, device=dev) if ids is None else ids.long()
        cols = torch.arange(n, device=dev) if cols is None else cols.long()
        valid = (ids >= 0) & (ids < self.n_envs) & (cols >= 0) & (cols < k)
        if snap.game != "space_invaders":
            tbl = data[_snap.TBL_WORD].long().index_select(0, cols.clamp(0, k - 1))
            valid &= (tbl >= 0) & (tbl < snap.table_count)
        order = torch.arange(n, device=dev)
        tgt = torch.where(valid, ids, self.n_envs)
        last = torch.full((self.n_envs + 1,), -1, dtype=torch.long, device=dev).scatter_reduce_(0, tgt, order, reduce="amax")
        sel = (valid & (last.index_select(0, tgt) == order)).nonzero().squeeze(1)
        self.obs.index_copy_(0, ids.index_select(0, sel), obs.index_select(0, cols.index_select(0, sel)))

    def fork(self, src_ids, dst_ids=None):
        """BatchedToybox.fork for wrapped envs, observation rings included."""
        snap = self.save_state(src_ids)
        dst = _snap.id_tensor(dst_ids, self.n_envs, self.device, "env id")
        self.load_state(snap, dst, _snap.fork_columns(snap.k, self.n_envs if dst is None else dst.numel(), self.device))

    def order(self):
        """ring slots, oldest observation first"""
        return [(self.slot + 1 + i) % self.k for i in range(self.k)]

    @property
    def channels(self):
        """bytes per observation pixel: 1 (gray) or 3 (RGB)"""
        return 1 if self.grayscale else 3

    def stacked(self):
        """FrameStack's observation (atari_wrappers.py:246-275) for every env, oldest first: uint8[N, out_h, out_w, k], or in
        colour uint8[N, out_h, out_w, 3k] with frame-major channels (the oldest frame's R, G, B first), the concatenation
        along the last axis that LazyFrames and VecFrameStack produce."""
        idx = torch.as_tensor(self.order(), device=self.device)
        ring = self.obs.index_select(1, idx)
        if self.grayscale:
            return ring.permute(0, 2, 3, 1).contiguous()
        return ring.permute(0, 2, 3, 1, 4).reshape(self.n_envs, self.out_h, self.out_w, 3 * self.k)


def _got_rings(snap):
    """what a refused snapshot holds, for the message"""
    if not getattr(snap, "wrapped", False):
        return " (got a snapshot of unwrapped envs)"
    sh = tuple(snap.obs.shape[1:])
    ch = sh[3] if len(sh) > 3 else 1
    return " (got %s rings of %d channel%s)" % (" x ".join(str(v) for v in sh[:3]), ch, "" if ch == 1 else "s")


class _Box:
    def __init__(self, low, high, shape, dtype):
        self.low, self.high, self.shape, self.dtype = low, high, tuple(shape), np.dtype(dtype)


class _Discrete:
    def __init__(self, n):
        self.n, self.shape, self.dtype = int(n), (), np.dtype(np.int64)


class ToyboxVecEnv:
    """The VecEnv surface of baselines (vec_env/__init__.py:26-131) over a DeepmindToybox: numpy in, numpy out, one
    process, one GPU.  It stands for `VecFrameStack(make_vec_env(env_id, 'atari', n, seed), 4)` (run.py:123-125): the stack
    of a finished env is zeroed and holds its reset observation only (vec_frame_stack.py:17-30), and
    `infos[i]['episode'] = {'r', 'l', 't'}` appears when env i's game ends (or its time limit, max_episode_steps, ends the
    episode; `infos[i]['TimeLimit.truncated'] = True` then, as gym's TimeLimit reports it), exactly as the Monitor between make_atari and
    wrap_deepmind reports it (bench/monitor.py:58-76: r = sum of raw rewards, l = MaxAndSkipEnv steps incl. those of
    FireResetEnv / EpisodicLifeEnv resets, t = seconds since start) -- both counters are kept by the step kernel.
    monitor_file: path of a Monitor-compatible CSV (bench/monitor.py:22-28,70-71,96-126: a '#{json header}' line, then the
    columns r,l,t), one row per finished episode."""

    def __init__(self, game, num_envs, monitor_file=None, **kw):
        kw.setdefault("stack_reset", "zero")
        self.env = DeepmindToybox(game, num_envs, **kw)
        self.num_envs = int(num_envs)
        e = self.env
        self.observation_space = _Box(0, 255, (e.out_h, e.out_w, e.channels * e.k), np.uint8)
        self.action_space = _Discrete(e.n_actions)
        self._actions = None
        self._t0 = time.time()
        self.closed = False
        self.episode_rewards, self.episode_lengths, self.episode_times = [], [], []
        self._csv = None
        if monitor_file is not None:
            if not monitor_file.endswith("monitor.csv"):
                monitor_file = monitor_file + ".monitor.csv" if not os.path.isdir(monitor_file) else os.path.join(monitor_file, "monitor.csv")
            self._csv = open(monitor_file, "wt")
            self._csv.write("#%s\n" % json.dumps({"t_start": self._t0, "env_id": "%sToyboxNoFrameskip-v4" % game.title().replace("_", "")}))
            self._csv.write("r,l,t\n")
            self._csv.flush()

    def reset(self):
        self.env.reset()
        return self.env.stacked().cpu().numpy()

    def step_async(self, actions):
        self._actions = np.ascontiguousarray(actions, dtype=np.int32)

    def step_wait(self):
        e = self.env
        e.step(self._actions)
        obs = e.stacked().cpu().numpy()
        rew = e.reward.cpu().numpy().astype(np.float32)
        done = e.done.cpu().numpy().astype(bool)
        real = e.real_done.cpu().numpy().astype(bool)
        trunc = e.truncated.cpu().numpy().astype(bool)
        score = e.score.cpu().numpy().astype(np.int64)
        lives = e.lives.cpu().numpy()
        infos = [{"lives": int(lives[i]), "score": int(score[i])} for i in range(self.num_envs)]
        for i in np.flatnonzero(trunc):
            infos[i]["TimeLimit.truncated"] = True
        ended = real | trunc
        if ended.any():
            ep_r, ep_l = e.ep_return.cpu().numpy(), e.ep_length.cpu().numpy()
            t = round(time.time() - self._t0, 6)
            for i in np.flatnonzero(ended):
                ep = {"r": round(float(ep_r[i]), 6), "l": int(ep_l[i]), "t": t}
                infos[i]["episode"] = ep
                self.episode_rewards.append(ep["r"])
                self.episode_lengths.append(ep["l"])
                self.episode_times.append(t)
                if self._csv is not None:
                    self._csv.write("%s,%d,%s\n" % (ep["r"], ep["l"], ep["t"]))
            if self._csv is not None:
                self._csv.flush()
        return obs, rew, done, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def close(self):
        if not self.closed:
            self.env.close()
            self.closed = True
            if self._csv is not None:
                self._csv.close()

    def get_episode_rewards(self):           # the Monitor accessors of bench/monitor.py:84-94
        return self.episode_rewards

    def get_episode_lengths(self):
        return self.episode_lengths

    def get_episode_times(self):
        return self.episode_times

    def get_images(self):
        return self.env.pool.render(obs="rgb").cpu().numpy()

    def render(self, mode="rgb_array"):
        return self.get_images()

    @property
    def unwrapped(self):
        return self
