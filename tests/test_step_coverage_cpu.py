"""CPU tier: the oracle side of the step-kernel coverage tests (step_coverage_ref) on its own.  The transition scenarios must
keep reaching their transitions (the GPU tests assert the same counts, so a change that stops a scenario short fails here
first), and the helpers that OracleBatch lacks must agree with OracleBatch where the two overlap: ALE ids, full-batch resets
and seeds, configs given at construction."""
import ctypes as C

import numpy as np
import pytest

import step_coverage_ref as R
from conftest import json_diff

GAMES = ["breakout", "amidar", "space_invaders"]


@pytest.mark.parametrize("name", list(R.SCENARIOS))
def test_scenario_reaches_its_transition(oracle_mod, name):
    want = R.SCENARIOS[name][-1]
    got = R.run_scenario(name)
    assert got == want, (name, got, want)
    assert max(got.values()) > 0


def _one_life(ref, every):
    for i in range(0, ref.n, every):
        js = ref.state_json(i)
        js["lives"] = 1
        ref.write_state(i, js)


@pytest.mark.parametrize("game", GAMES)
def test_input_step_and_statistics_match_batch_step(oracle_mod, game):
    """step_ale (ALE id -> mask -> step_inputs) == OracleBatch.step with auto-reset, frame by frame; the statistics
    accumulator == the episodes restated from OracleBatch's own rewards and dones"""
    n, seed0 = 24, 70
    ref = R.RefBatch(game, n, seed0)
    ob = oracle_mod.OracleBatch(game, n, seeds=seed0 + np.arange(n))
    _one_life(ref, 3)
    for i in range(0, n, 3):
        ob.write_state_json(i, ref.state_json(i))
    ret, length, eps = np.zeros(n, np.int64), np.zeros(n, np.int64), []
    for t in range(600):
        acts = R.random_actions(game, n, t, seed=31)
        got = ref.step_ale(acts, auto_reset=True)
        want = ob.step(acts, auto_reset=True)
        for g, w in zip(got, want):
            assert np.array_equal(g, w), t
        ret += want[0]
        length += 1
        for i in np.nonzero(want[1])[0]:
            eps.append((int(ret[i]), int(length[i])))
            ret[i] = length[i] = 0
    for i in range(n):
        assert json_diff(ref.state_json(i), ob.state_json(i)) == [], i
    assert len(eps) >= 4
    assert ref.read_stats() == [len(eps), sum(r for r, _ in eps), sum(l for _, l in eps), max(r for r, _ in eps)]
    assert ref.read_stats(reset=True)[0] == len(eps) and ref.read_stats() == [0, 0, 0, 0]


def test_masks_outside_the_ale_set(oracle_mod):
    """bits 6-7 and button2 reach no game: a mask steps like the mask without them (left+right, up+down and the rest are
    game rules, compared with the GPU in test_gpu_step_coverage)"""
    for game in GAMES:
        a, b = R.RefBatch(game, 16, 5), R.RefBatch(game, 16, 5)
        for t in range(400):
            m = (np.arange(16) * 37 + t * 11) % 256
            assert all(np.array_equal(x, y) for x, y in zip(a.step_inputs(m), b.step_inputs(m & 0x1F)))
        assert all(json_diff(a.state_json(i), b.state_json(i)) == [] for i in range(16)), game


@pytest.mark.parametrize("game", GAMES)
def test_resets_seeds_and_config_match_batch(oracle_mod, game):
    """new_game() over every env == OracleBatch.new_game; reseed of every env == OracleBatch.seed; write_config of a document
    == an OracleBatch built with it; a masked new_game touches only the flagged envs"""
    n = 9
    ref = R.RefBatch(game, n, 11)
    ob = oracle_mod.OracleBatch(game, n, seeds=11 + np.arange(n))
    ref.new_game()
    ob.new_game()
    assert all(json_diff(ref.state_json(i), ob.state_json(i)) == [] for i in range(n))
    ref.reseed(np.arange(n) + 500)
    ref.new_game()
    ob.seed(np.arange(n) + 500)
    assert all(json_diff(ref.state_json(i), ob.state_json(i)) == [] for i in range(n))
    cfg = ref.config_json()
    cfg["start_lives"] = 2
    ref.write_config(cfg)
    for _ in range(oracle_mod.NEW_GAMES_AT_CTOR[game]):       # as many as the OracleBatch constructor runs
        ref.new_game()
    ob2 = oracle_mod.OracleBatch(game, n, cfg_json=cfg)
    assert all(json_diff(ref.state_json(i), ob2.state_json(i)) == [] for i in range(n)) and int(ref.lives.min()) == 2
    before = [ref.state_json(i) for i in range(n)]
    for t in range(30):
        ref.step_ale(R.random_actions(game, n, t), auto_reset=False)
    stepped = [ref.state_json(i) for i in range(n)]
    fresh = oracle_mod.OracleBatch(game, n, cfg_json=cfg)
    C.memmove(fresh.sim, ref.b.sim, C.sizeof(fresh.sim))
    fresh.new_game()
    mask = np.arange(n) % 3 == 1
    ref.new_game(mask)
    for i in range(n):
        assert json_diff(ref.state_json(i), fresh.state_json(i) if mask[i] else stepped[i]) == [], i
        assert ref.ep_len[i] == (0 if mask[i] else 30)
    assert json_diff(before[0], stepped[0]) != []


def test_tracking_policy_restates_the_per_env_rule(oracle_mod):
    """the vectorised policy == the per-env restatement of test_gpu_parity's tracking test (on states with a ball)"""
    n = 40
    ref = R.RefBatch("breakout", n, 3)
    for t in range(1200):
        acts = R.breakout_tracking(ref, t)
        for i in range(n):
            s = ref.b.states[i]
            if s.is_dead:
                want = 1
            else:
                bx = s.balls[0].position.x + ((i * 7 + t // 50) % 9 - 4)
                want = 3 if bx > s.paddle.position.x + 1 else 4 if bx < s.paddle.position.x - 1 else 0
            assert acts[i] == want, (t, i)
        ref.step_ale(acts)
    assert int(ref.score.max()) > 20


def test_action_index_matches_oracle(oracle_mod):
    envs = np.arange(300)
    for seed, t, k in ((0xB200, 0, 4), (7, 12345, 18), (2 ** 64 - 1, 2 ** 40, 10)):
        got = R.action_index(seed, envs, t, k)
        assert list(got) == [oracle_mod.action_index(seed, int(e), t, k) for e in envs]
    assert C.sizeof(oracle_mod.Rng) == 16
