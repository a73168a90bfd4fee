"""TEST INFRASTRUCTURE: the oracle side of the step-kernel coverage tests (test_step_coverage_cpu.py, test_gpu_step_coverage.py).

RefBatch is oracle.OracleBatch with the pool operations OracleBatch lacks, each built from the oracle's existing ctypes functions:

  step_inputs      BatchedToybox.apply_action(Input masks): tbo_<game>_step per env with the raw mask, then the bookkeeping of
                   tbo_batch_step (reward = max(score - prev_score, 0), done = lives <= 0, auto-reset through new_game1)
  reseed           set_seed(seeds, env_ids): tbo_rng_seed on the listed envs' simulator rng
  new_game(mask)   new_game1 of oracle/batch.c on the flagged envs: a copy of the config whose rand is the env's simulator rng
  write_config     write_config_json: the codec into the shared config, then every simulator rng restarts from its rand
  set_score        set_property("score"): score and prev_score both take the value, as write_state_json does

and the episode statistics of the pool (episode_stats), restated in plain int64 Python: per env an episode length and return
that count every step (dead envs without auto-reset included), start again at new_game and survive state writes; an episode
ends where a step leaves done set and lives were above 0 before it; words: episodes, sum of returns, sum of lengths, max return.

The scenario builders put envs next to a transition -- Breakout's wall refill, Space Invaders' wave clear, Amidar's level
completion and chase -- by editing the state JSON; the same documents go into the pool.  The policies restate the action
rules the tests drive them with."""
import ctypes as C

import numpy as np

from oracle import oracle as O

STAGED = [None, "0", "1"]               # TBX_STEP_STAGED: the game's default step kernel, the lazy one, the staged one
M64 = (1 << 64) - 1


def action_index(seed, envs, t, n_legal):
    """oracle.action_index for many envs at once (tbx_action_index: the splitmix64 finaliser of (seed, env, t))"""
    with np.errstate(over="ignore"):
        z = np.uint64(seed & M64) + np.asarray(envs, np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64((t * 0xD1B54A32D192ED03) & M64)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (((z >> np.uint64(32)) * np.uint64(n_legal)) >> np.uint64(32)).astype(np.int64)


def random_actions(game, n, t, seed=0xB200):
    legal = np.asarray(O.LEGAL[game], np.int32)
    return legal[action_index(seed, np.arange(n), t, len(legal))]


class RefBatch:
    def __init__(self, game, n, seed0, cfg_json=None):
        self.b = O.OracleBatch(game, n, seeds=(seed0 + np.arange(n)) & 0xFFFFFFFF, cfg_json=cfg_json)
        self.game, self.n, self.L = game, n, self.b.L
        p = O.PREFIX[game]
        self._step, self._new = getattr(self.L, "tbo_%s_step" % p), getattr(self.L, "tbo_%s_new_game" % p)
        self.St = O.STATE[game]
        self.ss = C.sizeof(self.St)
        base = C.addressof(self.b.states)
        self.ptrs = [C.c_void_p(base + i * self.ss) for i in range(n)]
        self.score, self.lives, self.level = (self.view(lambda s: s, f) for f in ("score", "lives", "level"))
        self.ep_len = np.zeros(n, np.int64)
        self.ep_ret = np.zeros(n, np.int64)
        self.stats = np.zeros(4, np.int64)
        self._ale = [self.L.tbo_ale_action_to_input(a) for a in range(18)]

    def view(self, parent, field, dtype=np.int32):
        """a live numpy view of one scalar field of every env's state: `field` of the sub-struct parent(state)"""
        s0 = self.b.states[0]
        par = parent(s0)
        off = C.addressof(par) - C.addressof(self.b.states) + getattr(type(par), field).offset
        return np.ndarray((self.n,), dtype, buffer=self.b.states, offset=off, strides=(self.ss,))

    # ------------------------------------------------------------------ steps
    def step_inputs(self, masks, auto_reset=True):
        masks = np.asarray(masks)
        assert masks.shape == (self.n,)
        lives_before = self.lives.copy()
        cfg = C.byref(self.b.cfg)
        for i in range(self.n):
            self._step(cfg, self.ptrs[i], int(masks[i]))
        score, lives = self.score.copy(), self.lives.copy()
        reward = np.maximum(score - self.b.prev_score, 0)
        done = lives <= 0
        self.b.prev_score[:] = score
        self.ep_len += 1
        self.ep_ret += reward
        ended = done & (lives_before > 0)
        if ended.any():
            self.stats[0] += int(ended.sum())
            self.stats[1] += int(self.ep_ret[ended].sum())
            self.stats[2] += int(self.ep_len[ended].sum())
            self.stats[3] = max(int(self.stats[3]), int(self.ep_ret[ended].max()))
        if auto_reset and done.any():
            self.new_game(done)
        return reward.astype(np.int32), done, score, lives

    def step_ale(self, actions, auto_reset=True):
        return self.step_inputs([self._ale[int(a)] for a in actions], auto_reset)

    # ------------------------------------------------------------------ resets, seeds, config
    def new_game(self, mask=None):
        ids = range(self.n) if mask is None else np.nonzero(np.asarray(mask))[0]
        for i in ids:
            i = int(i)
            c = type(self.b.cfg).from_buffer_copy(self.b.cfg)
            c.rand = self.b.sim[i]
            self._new(C.byref(c), self.ptrs[i])
            self.b.sim[i] = c.rand
            self.b.prev_score[i] = self.score[i]
            self.ep_len[i] = self.ep_ret[i] = 0

    def reseed(self, seeds, ids=None):
        ids = range(len(seeds)) if ids is None else ids
        for s, i in zip(seeds, ids):
            self.L.tbo_rng_seed(C.byref(self.b.sim, int(i) * C.sizeof(O.Rng)), C.c_uint32(int(s) & 0xFFFFFFFF))

    def config_json(self):
        """config_to_json as the pool reports it: the rand is env 0's simulator rng"""
        js = O.CODEC[self.game][2](self.b.cfg)
        js["rand"] = {"state": [int(self.b.sim[0].s[0]), int(self.b.sim[0].s[1])]}
        return js

    def write_config(self, js):
        O.CODEC[self.game][3](self.b.cfg, js)
        for i in range(self.n):
            self.b.sim[i] = self.b.cfg.rand

    # ------------------------------------------------------------------ state edits
    def state_json(self, i):
        return self.b.state_json(i)

    def write_state(self, i, js):
        self.b.write_state_json(i, js)          # prev_score <- score; the episode counters stay

    def set_score(self, values, mask):
        m = np.asarray(mask, bool)
        self.score[m] = np.broadcast_to(np.asarray(values, np.int32), (self.n,))[m]
        self.b.prev_score[m] = self.score[m]

    def read_stats(self, reset=False):
        out = [int(v) for v in self.stats]
        if reset:
            self.stats[:] = 0
        return out

    def render(self, mode):
        return self.b.render(mode)


# ---------------------------------------------------------------------------------------------------------------------------
# policies
def breakout_tracking(ref, t):
    """fill_policy_actions(policy 1), as tbx_fill_actions_policy documents it: FIRE while the env waits for a serve, else move
    the paddle toward the first ball's x plus an aim offset ((env * 7 + t // 50) % 9) - 4 (RIGHT past paddle + 1, LEFT below
    paddle - 1, else NOOP).  The kernel reads ball slot 0 whatever the ball count."""
    if not hasattr(ref, "_trk"):
        ref._trk = (ref.view(lambda s: s, "is_dead", np.uint8), ref.view(lambda s: s.balls[0].position, "x", np.float64),
                    ref.view(lambda s: s.paddle.position, "x", np.float64))
    dead, bx, px = ref._trk
    off = ((np.arange(ref.n) * 7 + t // 50) % 9 - 4).astype(np.float64)
    aim = bx + off
    acts = np.where(aim > px + 1.0, 3, np.where(aim < px - 1.0, 4, 0))
    return np.where(dead != 0, 1, acts).astype(np.int32)


SI_SHOOTING = [11, 12, 1, 11, 12, 1, 3, 4]


def si_shooting(n, t):
    """the emulation tier's Space Invaders shooting policy, each env at its own phase"""
    return np.asarray([SI_SHOOTING[(t // 15 + i) % 8] for i in range(n)], np.int32)


# ---------------------------------------------------------------------------------------------------------------------------
# scenario builders: edit every env of `ref` next to a transition; return the documents (to be written into the pool too)
def _edit_all(ref, edit):
    docs = []
    for i in range(ref.n):
        js = ref.state_json(i)
        edit(js, i, np.random.default_rng(1000 + i))
        ref.write_state(i, js)
        docs.append(js)
    return docs


def breakout_near_refill(ref):
    """a few destructible bricks left in the lower rows, and two or three indestructible ones that the refill revives too"""
    def edit(js, i, g):
        bricks = js["bricks"]
        keep = set(int(k) for k in g.choice([b for b in range(len(bricks)) if bricks[b]["row"] >= 3], size=2 + i % 3, replace=False))
        hard = set(int(k) for k in g.choice([b for b in range(len(bricks)) if b not in keep], size=2 + i % 2, replace=False))
        for k, b in enumerate(bricks):
            b["alive"] = k in keep or k in hard or (i % 4 == 0 and k % 17 == 0 and k not in keep)
            if k in hard or (i % 4 == 0 and k % 17 == 0 and k not in keep):
                b["destructible"] = False
    return _edit_all(ref, edit)


def si_near_wave_clear(ref):
    """1-3 invaders left, drawn from both words of the alive mask (ids below and above 32)"""
    def edit(js, i, g):
        low = [int(k) for k in g.choice(32, size=1 + (i % 2), replace=False)]
        high = [32 + int(g.integers(4))] if i % 3 != 2 else []
        alive = set(low + high) if (low + high) else {int(g.integers(36))}
        for k, e in enumerate(js["enemies"]):
            e["alive"] = k in alive
    return _edit_all(ref, edit)


AMI_SEGMENT = [(31, y) for y in range(13, 18)]      # the inside of the column segment the player starts on, (31, 12) to (31, 18)


def _box_perimeter(b):
    (x0, y0), (x1, y1) = (b["top_left"]["tx"], b["top_left"]["ty"]), (b["bottom_right"]["tx"], b["bottom_right"]["ty"])
    return {(x, y) for x in range(x0, x1 + 1) for y in (y0, y1)} | {(x, y) for y in range(y0, y1 + 1) for x in (x0, x1)}


def _amidar_almost_painted(js, unpainted):
    """every walkable tile painted but `unpainted`; every box whose perimeter is then complete painted, except the chase corners"""
    tiles = js["board"]["tiles"]
    for y in range(31):
        for x in range(32):
            if tiles[y][x] != "Empty":
                tiles[y][x] = "Unpainted" if (x, y) in unpainted else "Painted"
    for b in js["board"]["boxes"]:
        b["painted"] = not b["triggers_chase"] and all(tiles[y][x] == "Painted" for x, y in _box_perimeter(b))


def amidar_near_level(ref):
    """painting the segment next to the player completes every box: the level ends in the frame the player closes it"""
    return _edit_all(ref, lambda js, i, g: _amidar_almost_painted(js, set(AMI_SEGMENT)))


AMI_BLOCKED_BOX = 14        # a non-corner box in the middle of the board


def amidar_near_chase(ref):
    """as amidar_near_level, but one non-corner box can never be finished (a tile of its perimeter is taken off the maze):
    painting the segment paints the four chase corners, chase starts and the level goes on.  Half the enemies hunt the player
    (EnemyTargetPlayer), so that catches happen within the chase."""
    def edit(js, i, g):
        box = js["board"]["boxes"][AMI_BLOCKED_BOX]
        assert not box["triggers_chase"]
        x0, y0 = box["top_left"]["tx"], box["top_left"]["ty"]
        x1 = box["bottom_right"]["tx"]
        hole = ((x0 + x1) // 2, y0)
        _amidar_almost_painted(js, set(AMI_SEGMENT))
        js["board"]["tiles"][hole[1]][hole[0]] = "Empty"
        box["painted"] = False
        js["chase_timer"] = 0
        for k, e in enumerate(js["enemies"]):
            if k % 2 == i % 2:
                e["ai"] = {"EnemyTargetPlayer": {"start": {"tx": 0, "ty": 0}, "start_dir": "Down", "vision_distance": 60, "dir": "Down",
                                                 "player_seen": None}}
    return _edit_all(ref, edit)


def amidar_wander(n, t):
    """the emulation tier's Amidar wandering policy, each env at its own phase"""
    dirs = [2, 3, 5, 4]
    return np.asarray([dirs[((t + 23 * i) // 37 + (t // 500)) % 4] if (t + i) % 211 else 1 for i in range(n)], np.int32)


# ---------------------------------------------------------------------------------------------------------------------------
# transition scenarios: (game, n, seed0, frames, builder, policy, how many envs reach each transition on the oracle).  The batch sizes straddle the
# staged kernel's envs per block (Breakout 128, Amidar and Space Invaders 32).
def _policy_tracking(ref, t):
    return breakout_tracking(ref, t)


def _policy_shooting(ref, t):
    return si_shooting(ref.n, t)


def _policy_random(ref, t):
    return random_actions(ref.game, ref.n, t)


SCENARIOS = {
    "breakout_refill": ("breakout", 129, 300, 2500, breakout_near_refill, _policy_tracking, {"level": 52}),
    "si_wave_clear": ("space_invaders", 65, 400, 1200, si_near_wave_clear, _policy_shooting, {"level": 46}),
    "amidar_level": ("amidar", 33, 500, 800, amidar_near_level, _policy_random,
                     {"level": 21, "chase_start": 0, "catch": 0, "chase_expiry": 0}),
    "amidar_chase": ("amidar", 31, 600, 900, amidar_near_chase, _policy_random,
                     {"level": 0, "chase_start": 25, "catch": 11, "chase_expiry": 21}),
}


class Events:
    """per-frame transition detection on the oracle's states: level ups, and Amidar's chase start, catches and chase expiry"""

    def __init__(self, ref):
        self.ref = ref
        self.counts = {"level": np.zeros(ref.n, bool)}
        if ref.game == "amidar":
            self.chase = ref.view(lambda s: s, "chase_timer")
            self.caught = [ref.view(lambda s, k=k: s.enemies[k], "caught", np.uint8) for k in range(O.AmiState.enemies.size // C.sizeof(O.AmiMob))]
            for k in ("chase_start", "catch", "chase_expiry"):
                self.counts[k] = np.zeros(ref.n, bool)

    def before(self):
        self.lv = self.ref.level.copy()
        if self.ref.game == "amidar":
            self.ct = self.chase.copy()
            self.nc = np.sum([c != 0 for c in self.caught], axis=0)

    def after(self, done):
        """the envs with a transition in this step (taken before an auto-reset replaces their state)"""
        ev = (self.ref.level > self.lv) & ~done
        self.counts["level"] |= ev
        if self.ref.game == "amidar":
            ct, nc = self.chase, np.sum([c != 0 for c in self.caught], axis=0)
            start, catch = (self.ct == 0) & (ct > 0) & ~done, (nc > self.nc) & ~done
            expiry = (self.ct > 0) & (ct == 0) & ~done & ~ev
            for k, v in (("chase_start", start), ("catch", catch), ("chase_expiry", expiry)):
                self.counts[k] |= v
            ev = ev | start | catch | expiry
        return ev

    def totals(self):
        return {k: int(v.sum()) for k, v in self.counts.items()}


def run_scenario(name, hook=None):
    """plays scenario `name` on the oracle with auto-reset; hook(ref, docs) is called once after the build and returns a
    per-frame callback f(t, actions, (reward, done, score, lives), events) run after every oracle step (the GPU mirror).
    Returns the counts of envs that reached each transition."""
    game, n, seed0, frames, build, policy, _ = SCENARIOS[name]
    ref = RefBatch(game, n, seed0)
    docs = build(ref)
    per_frame = hook(ref, docs) if hook else None
    ev = Events(ref)
    for t in range(frames):
        acts = policy(ref, t)
        ev.before()
        out = ref.step_ale(acts, auto_reset=False)
        events = ev.after(out[1])
        if out[1].any():                        # auto-reset after the transition check
            ref.new_game(out[1])
        if per_frame:
            per_frame(t, acts, out, events)
    return ev.totals()
