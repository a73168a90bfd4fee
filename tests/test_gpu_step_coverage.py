"""GPU tier: the step kernels beyond random play, against the oracle-side mirror of step_coverage_ref, bit for bit on the same
seeds and inputs.  Every test runs with TBX_STEP_STAGED unset (the game's default kernel), "0" (step_kernel, records read in
place from the word-major planes) and "1" (step_staged_kernel, records staged through shared memory), at batch sizes that
straddle a warp and the staged kernel's envs per block (Breakout 128, Amidar and Space Invaders 32).  Every frame compares
reward, done, score, lives and level; the full state JSON and the frames are compared at intervals and at every transition.

Covered: Breakout's wall refill (driven by fill_policy_actions, checked against its rule every frame), Space Invaders' wave
clear, Amidar's level completion, chase start, catches and chase expiry; apply_action with every uint8 mask, auto-reset on
and off; config edits written mid-rollout, then some envs continued and the others restarted by a masked new_game; state
interventions incl. several Breakout balls lost in one frame and a ball that hits the 64-slice cap; set_seed with env ids;
get_level / game_over; all four episode-statistics words, their reset and the device copy; the Breakout column operations on
edited brick tables."""
import numpy as np
import pytest
import torch

import step_coverage_ref as R
from conftest import json_diff

pytestmark = pytest.mark.gpu
GAMES = ["breakout", "amidar", "space_invaders"]


@pytest.fixture(params=R.STAGED, ids=lambda v: "default" if v is None else "staged" + v)
def staged(request, monkeypatch):
    """the step kernel variant: TBX_STEP_STAGED is read at every launch"""
    if request.param is None:
        monkeypatch.delenv("TBX_STEP_STAGED", raising=False)
    else:
        monkeypatch.setenv("TBX_STEP_STAGED", request.param)
    return request.param


class Mirror:
    """a pool and its oracle mirror built from the same seeds"""

    def __init__(self, tbx, ref, seed0):
        self.ref, self.n = ref, ref.n
        self.pool = tbx.BatchedToybox(ref.game, ref.n, seeds=seed0)
        self.dev = self.pool.device

    def write_states(self, docs, ids=None):
        self.pool.write_state_json(docs, ids)

    def check_step(self, out, t):
        """the step's outputs, then the scalars of the state after it (auto-reset included)"""
        p, ref = self.pool, self.ref
        r, d, s, l = out
        got = (p.reward.cpu().numpy(), p.done.cpu().numpy().astype(bool), p.score.cpu().numpy(), p.lives.cpu().numpy())
        for name, g, w in zip(("reward", "done", "score", "lives"), got, (r, d, s, l)):
            bad = np.nonzero(g != w)[0]
            assert bad.size == 0, (t, name, bad[:6], g[bad[:6]], w[bad[:6]])
        score, lives, level = (x.cpu().numpy() for x in p._scalars())
        assert np.array_equal(level, ref.level), (t, "level", np.nonzero(level != ref.level)[0][:6])
        assert np.array_equal(score, ref.score) and np.array_equal(lives, ref.lives), (t, "scalars")
        assert np.array_equal(p.game_over().cpu().numpy(), ref.lives <= 0), t

    def check_full(self, t, ids=None, modes=("rgba", "gray84")):
        ids = list(range(self.n)) if ids is None else [int(i) for i in ids]
        if ids:
            for i, js in zip(ids, self.pool.to_state_json(ids)):
                assert json_diff(js, self.ref.state_json(i)) == [], (t, i, json_diff(js, self.ref.state_json(i)))
        for mode in modes:
            got = self.pool.render(obs=mode).cpu().numpy().reshape(self.n, -1)
            want = self.ref.render(mode).reshape(self.n, -1)
            bad = np.argwhere(got != want)
            assert bad.size == 0, (t, mode, bad[:4])

    def step_ale(self, acts, t, auto_reset=True):
        out = self.ref.step_ale(acts.cpu().numpy() if torch.is_tensor(acts) else np.asarray(acts), auto_reset)
        self.pool.apply_ale_action(acts, auto_reset=auto_reset)
        self.check_step(out, t)
        return out

    def step_inputs(self, masks, t, auto_reset=True):
        out = self.ref.step_inputs(masks, auto_reset)
        self.pool.apply_action(torch.as_tensor(masks, dtype=torch.uint8), auto_reset=auto_reset)
        self.check_step(out, t)
        return out

    def policy_actions(self, t):
        """fill_policy_actions(policy 1) on the pool == the documented rule on the oracle's states"""
        acts = torch.empty(self.n, dtype=torch.int32, device=self.dev)
        self.pool.fill_policy_actions(acts, 1, t)
        want = R.breakout_tracking(self.ref, t)
        got = acts.cpu().numpy()
        assert np.array_equal(got, want), (t, np.nonzero(got != want)[0][:6])
        return acts

    def check_stats(self, t):
        want = self.ref.read_stats()
        assert self.pool.episode_stats() == want, (t, self.pool.episode_stats(), want)
        dev = torch.full((4,), -7, dtype=torch.int64, device=self.dev)
        self.pool.episode_stats_into(dev)
        assert dev.cpu().tolist() == want, t

    def close(self):
        self.pool.close()


# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(R.SCENARIOS))
def test_transition(tbx, staged, name):
    game, n, seed0, frames, _, _, want = R.SCENARIOS[name]
    box = {}

    def hook(ref, docs):
        m = box["m"] = Mirror(tbx, ref, seed0)
        m.write_states(docs)
        m.check_full(-1)

        def per_frame(t, acts, out, events):
            # the pool still holds the state the oracle stepped from, and `acts` is the policy's choice on it
            a = acts
            if game == "breakout":
                a = torch.empty(n, dtype=torch.int32, device=m.dev)
                m.pool.fill_policy_actions(a, 1, t)
                assert np.array_equal(a.cpu().numpy(), acts), (t, np.nonzero(a.cpu().numpy() != acts)[0][:6])
            m.pool.apply_ale_action(a, auto_reset=True)
            m.check_step(out, t)
            ids = np.nonzero(events)[0]
            if ids.size or t % 300 == 0:
                m.check_full(t, ids if t % 300 else None, modes=("rgb", "gray84"))
        return per_frame

    got = R.run_scenario(name, hook)
    assert got == want, (name, got, want)
    box["m"].check_full("end")
    box["m"].check_stats("end")
    box["m"].close()


# ---------------------------------------------------------------------------------------------------------------------------
MASK_N = {"breakout": 200, "amidar": 65, "space_invaders": 1}


@pytest.mark.parametrize("game", GAMES)
def test_every_input_mask(tbx, staged, game):
    """apply_action with every uint8 value (left+right, up+down, button2 and bits 6-7 included), auto-reset on and off in
    turns; a third of the envs start with one life so that games end inside the run"""
    n, seed0 = MASK_N[game], 40
    ref = R.RefBatch(game, n, seed0)
    m = Mirror(tbx, ref, seed0)
    docs = []
    for i in range(n):
        js = ref.state_json(i)
        if i % 3 == 0:
            js["lives"] = 1
        ref.write_state(i, js)
        docs.append(js)
    m.write_states(docs)
    perm = np.random.default_rng(5).permutation(256)
    seen = np.zeros(256, bool)
    for t in range(768):
        masks = perm[(t + 37 * np.arange(n)) % 256].astype(np.uint8)
        seen[masks] = True
        m.step_inputs(masks, t, auto_reset=(t // 64) % 2 == 0)
        if t % 192 == 0:
            m.check_full(t)
    assert seen.all()
    m.check_full("end", modes=("rgba", "rgb", "gray", "gray84"))
    m.check_stats("end")
    assert ref.stats[0] > 0
    m.close()


# ---------------------------------------------------------------------------------------------------------------------------
CONFIG_EDITS = {
    "breakout": [dict(paddle_discrete_segments=1, ball_speed_slow=3.0, ball_speed_fast=5.5, ball_speed_row_depth=1, row_scores=[9, 9, 5, 5, 2, 2]),
                 dict(paddle_discrete_segments=16, start_lives=2, ball_speed_slow=1.25, ball_speed_row_depth=5),
                 dict(paddle_discrete_segments=7, ball_speed_fast=3.0, bg_color={"r": 10, "g": 20, "b": 30, "a": 255})],
    "amidar": [dict(start_lives=1, start_jumps=2, chase_time=20, jump_time=10, box_bonus=7, chase_score_bonus=33),
               dict(start_lives=2, chase_time=5, jump_time=3, box_bonus=0, chase_score_bonus=250)],
    "space_invaders": [dict(start_lives=1, jitter=0.1, enemy_protocol="Random", row_scores=[1, 2, 3, 4, 5, 6]),
                       dict(start_lives=2, jitter=0.9, enemy_protocol="TargetPlayer"),
                       dict(jitter=0.0, row_scores=[60, 50, 40, 30, 20, 10])],
}
CONFIG_BUILD = {"breakout": (R.breakout_near_refill, 65), "amidar": (R.amidar_near_chase, 129),
                "space_invaders": (R.si_near_wave_clear, 33)}


@pytest.mark.parametrize("game", GAMES)
def test_edited_configs_mid_rollout(tbx, staged, game):
    """the scenario states of the game, played under a sequence of config edits written mid-rollout (the device copies of the
    config and the geometry tables); after each write a third of the envs restart through a masked new_game, the others go on"""
    build, n = CONFIG_BUILD[game]
    seed0 = 900
    ref = R.RefBatch(game, n, seed0)
    m = Mirror(tbx, ref, seed0)
    m.write_states(build(ref))
    t, top = 0, 1
    chase = ref.view(lambda s: s, "chase_timer") if game == "amidar" else None
    for k, edit in enumerate(CONFIG_EDITS[game] + [None]):
        for _ in range(250):
            if game == "breakout":
                acts = m.policy_actions(t)
            elif game == "space_invaders":
                acts = R.si_shooting(n, t)
            else:
                acts = R.random_actions(game, n, t, seed=k)
            out = ref.step_ale(np.asarray(acts.cpu() if torch.is_tensor(acts) else acts), True)
            m.pool.apply_ale_action(acts, auto_reset=True)
            m.check_step(out, t)
            top = max(top, int(ref.level.max()), 2 if chase is not None and chase.max() > 0 else 1)
            t += 1
        if edit is None:
            break
        assert json_diff(m.pool.config_to_json(), ref.config_json()) == [], (k, json_diff(m.pool.config_to_json(), ref.config_json()))
        cfg = ref.config_json()
        cfg.update(edit)
        m.pool.write_config_json(cfg)
        ref.write_config(cfg)
        assert json_diff(m.pool.config_to_json(), ref.config_json()) == [], k
        mask = (np.arange(n) + k) % 3 == 0
        m.pool.new_game(torch.as_tensor(mask))
        ref.new_game(mask)
        m.check_full(("config", k), modes=("rgb", "gray84"))
    m.check_full("end")
    m.check_stats("end")
    assert top > 1                  # a level went up (Amidar: a chase ran) under an edited config
    m.close()


# ---------------------------------------------------------------------------------------------------------------------------
def _brk_balls(js, i, g):
    """2-4 balls in play: those at even slots leave the field in the same frame (the survivors are compacted), the others fly up"""
    k = 2 + i % 3
    js["balls"] = [{"position": {"x": 40.0 + 45.0 * b, "y": 157.0}, "velocity": {"x": 0.5, "y": 3.0}} if b % 2 == 0 else
                   {"position": {"x": 30.0 + 50.0 * b, "y": 100.0}, "velocity": {"x": 1.25 * (b - 2), "y": -2.0}} for b in range(k)]
    js["is_dead"] = js["reset"] = False


def _brk_fast(js, i, g):
    """a ball that needs more than 64 slices of one radius per frame: the step stops at the cap"""
    js["balls"] = [{"position": {"x": 120.0, "y": 110.0}, "velocity": {"x": 151.0 + i, "y": -173.5}}]
    js["is_dead"] = js["reset"] = False


INTERVENTIONS = {   # test_emu_parity.test_interventions_step_like_oracle's edits, and the Breakout ball edits
    "breakout": [lambda js, i, g: (js["bricks"][5].update(alive=False), js["bricks"][30].update(color={"r": 9, "g": 8, "b": 7, "a": 255}),
                                   js["bricks"][31].update(destructible=False), js["bricks"][32]["position"].update(x=100.5),
                                   js["balls"].append({"position": {"x": 60.0, "y": 90.0}, "velocity": {"x": -1.5, "y": -1.5}}),
                                   js.update(paddle_width=48.0, lives=2)),
                 _brk_balls, _brk_fast],
    "amidar": [lambda js, i, g: (js.update(jumps=2, chase_timer=50), js["enemies"].pop(),
                                 js["enemies"][0].update(ai={"EnemyTargetPlayer": {"start": {"tx": 0, "ty": 0}, "start_dir": "Down", "vision_distance": 15,
                                                                                  "dir": "Down", "player_seen": None}}),
                                 js["enemies"][1].update(ai={"EnemyAmidarMvmt": {"vert": "Down", "horiz": "Right", "start_vert": "Down",
                                                                                "start_horiz": "Right", "start": {"tx": 0, "ty": 0}}}),
                                 js["enemies"][2].update(ai={"EnemyPerimeterAI": {"start": {"tx": 0, "ty": 0}}}),
                                 js["enemies"][3].update(ai={"EnemyRandomMvmt": {"start": {"tx": 31, "ty": 30}, "start_dir": "Up", "dir": "Up"}},
                                                         position={"x": 1984, "y": 2400}),
                                 js["player"]["position"].update(x=1000, y=480))],
    "space_invaders": [lambda js, i, g: (js.update(lives=1, enemy_shot_delay=2), js["ufo"].update(appearance_counter=1),
                                         js["shields"][1]["data"][3][4].update(a=0), js["enemies"][35].update(alive=False),
                                         js["ship"].update(x=100, color={"r": 1, "g": 2, "b": 3, "a": 255}))],
}
INTERVENTION_N = {"breakout": 129, "amidar": 31, "space_invaders": 65}


@pytest.mark.parametrize("game", GAMES)
def test_interventions_step_alike(tbx, staged, game):
    n, seed0 = INTERVENTION_N[game], 77
    ref = R.RefBatch(game, n, seed0)
    m = Mirror(tbx, ref, seed0)
    for t in range(300):
        m.step_ale(R.random_actions(game, n, t, seed=3), t)
    edits = INTERVENTIONS[game]
    ids = [i for i in range(n) if i % 4 != 3]               # every fourth env plays on unedited
    docs = []
    for i in ids:
        js = ref.state_json(i)
        edits[i % len(edits)](js, i, np.random.default_rng(i))
        ref.write_state(i, js)
        docs.append(js)
    m.write_states(docs, ids)
    m.check_full("edit", modes=("rgba",))
    nballs = ref.view(lambda s: s, "n_balls") if game == "breakout" else None
    compacted = 0
    for t in range(1200):
        before = nballs.copy() if nballs is not None else None
        acts = m.policy_actions(t) if game == "breakout" else R.random_actions(game, n, t, seed=4)
        out = ref.step_ale(np.asarray(acts.cpu() if torch.is_tensor(acts) else acts), True)
        m.pool.apply_ale_action(acts, auto_reset=True)
        m.check_step(out, t)
        if before is not None:
            compacted += int(np.sum((before >= 2) & (before - nballs >= 2) & (nballs > 0) & ~out[1]))
        if t < 8 or t % 200 == 0:
            m.check_full(t, [0, 1, 2, n - 1], modes=("rgba",) if t % 200 == 0 else ())
    m.check_full("end", modes=("rgba", "gray84"))
    m.check_stats("end")
    if game == "breakout":
        assert compacted > 0          # two balls or more left the field in one frame while others stayed in play
    m.close()


# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("game", GAMES)
def test_seed_ids_and_masked_new_game(tbx, staged, game):
    """set_seed(seeds, env_ids) reseeds only the listed envs' simulator rng; a masked new_game restarts only the flagged
    envs; the auto-resets that follow draw from the new rngs"""
    n, seed0 = {"breakout": 31, "amidar": 65, "space_invaders": 129}[game], 60
    ref = R.RefBatch(game, n, seed0)
    m = Mirror(tbx, ref, seed0)
    for t in range(100):
        m.step_ale(R.random_actions(game, n, t, seed=8), t)
    ids = np.random.default_rng(3).permutation(n)[: max(1, n // 2)]
    seeds = (np.arange(ids.size) * 2654435761 + 17) & 0xFFFFFFFF
    m.pool.set_seed(seeds.astype(np.uint32), env_ids=ids)
    ref.reseed(seeds, ids)
    mask = (np.arange(n) % 2 == 0) | (np.arange(n) == n - 1)
    m.pool.new_game(torch.as_tensor(mask))
    ref.new_game(mask)
    m.check_full("reseed")
    assert json_diff(m.pool.config_to_json(), ref.config_json()) == []
    docs = []
    for i in range(n):                                      # short games: the auto-resets below use the new rngs
        js = ref.state_json(i)
        js["lives"] = 1
        ref.write_state(i, js)
        docs.append(js)
    m.write_states(docs)
    for t in range(100, 700):
        m.step_ale(R.random_actions(game, n, t, seed=8), t)
    m.check_full("end")
    m.check_stats("end")
    assert ref.stats[0] > 0
    m.close()


# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("game", GAMES)
def test_episode_statistics(tbx, staged, game):
    """all four words of episode_stats against the accumulator: envs stepped after game over (auto-reset off in turns), JSON
    writes that set lives to 0, set_property('score'); episode_stats(reset=True) zeroes the counters; episode_stats_into
    copies the same words on the device"""
    n, seed0 = {"breakout": 129, "amidar": 33, "space_invaders": 65}[game], 20
    ref = R.RefBatch(game, n, seed0)
    m = Mirror(tbx, ref, seed0)
    docs = []
    for i in range(n):
        js = ref.state_json(i)
        js["lives"] = 1 if i % 4 == 0 else js["lives"]
        ref.write_state(i, js)
        docs.append(js)
    m.write_states(docs)
    m.check_stats("start")
    before_reset = None
    for t in range(900):
        if t == 380:                                        # game over written into a quarter of the envs, auto-reset off
            ids = [i for i in range(n) if i % 4 == 1]
            docs = []
            for i in ids:
                js = ref.state_json(i)
                js["lives"] = 0
                ref.write_state(i, js)
                docs.append(js)
            m.write_states(docs, ids)
        if t == 450:
            mask = np.arange(n) % 5 == 2
            vals = (np.arange(n) * 13 + 1000).astype(np.int32)
            m.pool.set_property("score", vals, mask)
            ref.set_score(vals, mask)
        if t == 600:
            before_reset = ref.read_stats(reset=True)
            assert m.pool.episode_stats(reset=True) == before_reset
            m.check_stats("reset")
        acts = R.random_actions(game, n, t, seed=12)
        acts[np.arange(n) % 7 == 3] = 1                       # FIRE: Breakout serves, so lives go
        m.step_ale(acts, t, auto_reset=(t // 75) % 2 == 0)
        if t % 50 == 49:
            m.check_stats(t)
    assert before_reset[0] > 0 and ref.stats[0] > 0, (before_reset, ref.stats)
    m.check_full("end", modes=("gray84",))
    m.close()


# ---------------------------------------------------------------------------------------------------------------------------
def test_breakout_columns_on_edited_brick_tables(tbx, staged):
    """breakout_fill_column / breakout_add_channel / breakout_channel_count on envs whose brick tables were edited through
    JSON (moved columns, columns outside 0..63, fewer bricks), against the same edits made through the oracle's JSON"""
    from toybox_b200 import interventions as IV
    n, seed0 = 33, 8
    ref = R.RefBatch("breakout", n, seed0)
    m = Mirror(tbx, ref, seed0)
    g = np.random.default_rng(4)
    docs = []
    for i in range(n):
        js = ref.state_json(i)
        kind = i % 5
        for k, b in enumerate(js["bricks"]):
            b["alive"] = bool(g.integers(4) > 0)
            if kind == 1:
                b["col"] = (b["col"] + 3) % 18                  # columns renumbered
            elif kind == 2:
                b["col"] = b["col"] + 50 if k % 2 else -1       # columns past 63 and negative: never counted
            elif kind == 3:
                b["col"] = b["row"]                             # rows as columns: six columns of 18 bricks
        if kind == 4:
            js["bricks"] = js["bricks"][: 40 + i]
        ref.write_state(i, js)
        docs.append(js)
    m.write_states(docs)

    def edit_ref(col, alive, mask):
        for i in np.nonzero(mask)[0]:
            js = ref.state_json(int(i))
            for b in js["bricks"]:
                if b["col"] == col:
                    b["alive"] = alive
            ref.write_state(int(i), js)

    def channels():
        out = np.zeros(n, np.int32)
        for i in range(n):
            cols = {}
            for b in ref.state_json(i)["bricks"]:
                if 0 <= b["col"] <= 63:
                    cols[b["col"]] = cols.get(b["col"], False) or b["alive"]
            out[i] = sum(1 for v in cols.values() if not v)
        return out

    for step, (col, alive) in enumerate([(3, False), (3, True), (5, False), (53, False), (2, True), (0, False), (17, False)]):
        mask = (np.arange(n) + step) % 3 != 0
        (IV.breakout_fill_column if alive else IV.breakout_add_channel)(m.pool, col, torch.as_tensor(mask))
        edit_ref(col, alive, mask)
        m.check_full(("column", col), modes=())
        want = channels()
        assert np.array_equal(IV.breakout_channel_count(m.pool).cpu().numpy(), want), (col, alive)
    assert channels().max() > 0
    for t in range(300):
        m.step_ale(m.policy_actions(t), t)
    m.check_full("end", modes=("rgba", "gray84"))
    m.close()
