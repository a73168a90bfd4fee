"""GPU tier: sticky actions and the episode time limit of the fused wrapper stack (DeepmindToybox(repeat_action_probability,
sticky_seed, max_episode_steps), tbx_wrap_set_sticky_actions / tbx_wrap_set_time_limit) against the oracle-side chain with
StickyActionEnv and TimeLimit (wrapped_protocol_ref.ProtocolWrappedEnv), env by env and bit for bit: stacked observations, rewards,
dones, real dones, truncation flags, lives, scores and Monitor's episode records.

Covered: p = 0.25 on the three games; sticky with the wrapper switches off, frame skip 1 and 3 and both stack modes; sticky
colour observations; p = 1; a short limit with and without sticky, through many truncations and some game overs; the VecEnv
infos and Monitor CSV; snapshots of a sticky wrap and loads across sticky and plain wraps; argument refusals."""
import ctypes as C

import numpy as np
import pytest

import wrapped_protocol_ref as R

pytestmark = pytest.mark.gpu
GAMES = ["breakout", "amidar", "space_invaders"]


def _one_life(js, i):
    """one life left in every other env: random play then ends whole games within a short limit"""
    if i % 2 == 0:
        js["lives"] = 1


def _run(game, n, steps, kw, seed0=500, grayscale=True, edit=None, probe=None):
    """the loop of test_gpu_wrappers._run, extended by the truncation flag; edit(js, i) is written into both sides after the
    reset; probe(env, refs) runs after every step.  Returns (agent dones, game overs, truncations)."""
    import torch
    from oracle import oracle as O
    from toybox_b200.wrappers import DeepmindToybox
    env = DeepmindToybox(game, n, seeds=seed0, noop_seed=7, grayscale=grayscale, **kw)
    refs = [R.ProtocolWrappedEnv(game, seed0 + i, env_id=i, noop_seed=7, **kw) for i in range(n)]
    if not grayscale:
        refs = [R.colour(r, kw.get("size", (84, 84))) for r in refs]
    n_act = env.n_actions
    obs = env.reset()
    want = np.stack([r.reset() for r in refs])
    assert np.array_equal(obs[:, env.order()].cpu().numpy(), want), "reset"
    if edit is not None:
        states = []
        for i, r in enumerate(refs):
            js = r.base.b.state_json(0)
            edit(js, i)
            r.base.b.write_state_json(0, js)
            states.append(js)
        env.pool.write_state_json(states)
    ndone = nreal = ntrunc = 0
    for t in range(steps):
        acts = np.asarray([O.action_index(0xB200, i, t, n_act) for i in range(n)], np.int32)
        obs, rew, done, info = env.step(torch.as_tensor(acts, device=env.device))
        got = obs[:, env.order()].cpu().numpy()
        rew, done = rew.cpu().numpy(), done.cpu().numpy().astype(bool)
        lives, score = info["lives"].cpu().numpy(), info["score"].cpu().numpy()
        real, trunc = info["real_done"].cpu().numpy().astype(bool), info["truncated"].cpu().numpy().astype(bool)
        ep_r, ep_l = info["ep_return"].cpu().numpy(), info["ep_length"].cpu().numpy()
        for i, r in enumerate(refs):
            w_obs, w_rew, w_done, w_info = r.step(int(acts[i]))
            assert (w_rew, w_done, w_info["lives"], w_info["score"], w_info["real_done"], w_info["truncated"]) == \
                (rew[i], done[i], lives[i], score[i], real[i], trunc[i]), (game, t, i, w_rew, rew[i], w_done, done[i], w_info, real[i], trunc[i])
            assert ("episode" in w_info) == bool(real[i] or trunc[i]), (game, t, i)
            if "episode" in w_info:
                assert (w_info["episode"]["r"], w_info["episode"]["l"]) == (ep_r[i], ep_l[i]), (game, t, i, w_info["episode"], ep_r[i], ep_l[i])
            bad = np.argwhere(got[i] != w_obs)
            assert bad.size == 0, (game, t, i, bad[:4], got[i][tuple(bad[0])], w_obs[tuple(bad[0])])
            ndone += int(w_done)
            nreal += int(real[i])
            ntrunc += int(trunc[i])
        if probe is not None:
            probe(env, refs)
    env.check()
    env.close()
    return ndone, nreal, ntrunc


@pytest.mark.parametrize("game", GAMES)
def test_sticky_rollout_bit_exact(game):
    nd, _, nt = _run(game, 12, 220 if game == "breakout" else 120, dict(repeat_action_probability=0.25))
    assert nt == 0
    if game == "breakout":
        assert nd > 0          # lost lives: the reset chains run sticky frames too


def test_sticky_wrapper_switches():
    p = dict(repeat_action_probability=0.25)
    _run("breakout", 6, 300, dict(p, episode_life=False, fire_reset=False, noop_max=0, frame_skip=1, stack_reset="zero"),
         edit=_one_life)
    _run("breakout", 6, 160, dict(p, episode_life=False, fire_reset=False, noop_max=0, frame_skip=3))
    _run("space_invaders", 4, 80, dict(p, frame_skip=3, noop_max=3, frame_stack=2, stack_reset="zero", sticky_seed=99))
    _run("amidar", 4, 80, dict(p, frame_skip=1, sticky_seed=7))                    # sticky_seed == noop_seed


def test_sticky_colour():
    _run("breakout", 6, 160, dict(repeat_action_probability=0.25), grayscale=False, edit=_one_life)


def test_always_sticky():
    """p = 1: no requested action ever takes effect, so Breakout's paddle stays where the game put it"""
    xs = []

    def probe(env, refs):
        xs.append(env.pool.get_property("paddle.position.x").cpu().numpy())

    _run("breakout", 8, 120, dict(repeat_action_probability=1.0), probe=probe)
    assert all(np.array_equal(x, xs[0]) for x in xs)
    _run("space_invaders", 4, 60, dict(repeat_action_probability=1.0))


@pytest.mark.parametrize("kw", [dict(max_episode_steps=37), dict(max_episode_steps=37, repeat_action_probability=0.25)])
def test_time_limit(kw):
    nd, nreal, nt = _run("breakout", 10, 260, kw, edit=_one_life)
    assert nt >= 20 and nreal >= 3, (nt, nreal)
    _run("space_invaders", 4, 90, dict(kw, max_episode_steps=23, frame_skip=3))


def test_vec_env_infos_and_csv(tmp_path):
    """infos[i]['episode'] where the game ended or the limit truncated it, infos[i]['TimeLimit.truncated'], and the Monitor CSV
    rows of both, against the oracle-side chain"""
    from oracle import oracle as O
    from toybox_b200.wrappers import ToyboxVecEnv
    n, kw = 8, dict(repeat_action_probability=0.25, max_episode_steps=45)
    path = str(tmp_path / "0")
    venv = ToyboxVecEnv("breakout", n, seeds=40, noop_seed=9, monitor_file=path, **kw)
    refs = [R.ProtocolWrappedEnv("breakout", 40 + i, env_id=i, noop_seed=9, stack_reset="zero", **kw) for i in range(n)]
    obs = venv.reset()
    assert np.array_equal(obs, np.stack([r.reset() for r in refs]).transpose(0, 2, 3, 1))
    rows, ntrunc = [], 0
    for t in range(300):
        acts = np.asarray([O.action_index(0xB200, i, t, 4) for i in range(n)], np.int32)
        obs, rew, done, infos = venv.step(acts)
        for i, r in enumerate(refs):
            w_obs, w_rew, w_done, w_info = r.step(int(acts[i]))
            assert np.array_equal(obs[i], w_obs.transpose(1, 2, 0)) and w_rew == rew[i] and w_done == done[i], (t, i)
            assert infos[i].get("TimeLimit.truncated", False) == w_info["truncated"], (t, i)
            assert ("episode" in infos[i]) == ("episode" in w_info), (t, i)
            if "episode" in w_info:
                assert (infos[i]["episode"]["r"], infos[i]["episode"]["l"]) == (w_info["episode"]["r"], w_info["episode"]["l"]), (t, i)
                rows.append((w_info["episode"]["r"], w_info["episode"]["l"]))
            ntrunc += int(w_info["truncated"])
    venv.close()
    assert ntrunc > 0 and rows and venv.get_episode_lengths() == [l for _, l in rows]
    lines = open(path + ".monitor.csv").read().splitlines()
    assert lines[1] == "r,l,t"
    assert [(float(x.split(",")[0]), int(x.split(",")[1])) for x in lines[2:]] == [(float(r), l) for r, l in rows]


@pytest.mark.parametrize("game", GAMES)
def test_sticky_snapshots(game):
    import torch
    from toybox_b200 import _lib
    from toybox_b200.wrappers import DeepmindToybox
    n, K = 24, 50
    env = DeepmindToybox(game, n, seeds=12, noop_seed=3, repeat_action_probability=0.25, max_episode_steps=30)
    rec = env.L.tbx_state_rows(env.pool._h)
    env.reset()
    gen = np.random.default_rng(0)
    for _ in range(40):
        env.step(torch.as_tensor(gen.integers(0, env.n_actions, n), dtype=torch.int32, device=env.device))
    snap = env.save_state()
    assert snap.wrapped and snap.rows == rec + 7
    words = snap.data[rec:].cpu().numpy()
    assert (words[6] > 0).all() and set(np.unique(words[5])) <= set(env.pool.get_legal_action_set())   # counter, ALE id
    stacked0 = env.stacked().cpu().numpy()
    acts = [torch.as_tensor(gen.integers(0, env.n_actions, n), dtype=torch.int32, device=env.device) for _ in range(K)]

    def run():
        out = []
        for a in acts:
            _, r, d, info = env.step(a)
            out += [env.stacked().cpu().numpy()] + [x.cpu().numpy().copy() for x in (r, d, info["real_done"], info["truncated"],
                                                                                       info["ep_return"], info["ep_length"])]
        return out

    first = run()
    assert any(x.any() for x in first[4::7])               # the 50 steps truncate some episodes
    env.load_state(snap)
    env.check()
    assert np.array_equal(env.stacked().cpu().numpy(), stacked0)
    second = run()
    assert len(first) == len(second) and all(np.array_equal(a, b) for a, b in zip(first, second))

    # a plain wrap refuses the sticky snapshot and the reverse, and neither pool changes
    plain = DeepmindToybox(game, n, seeds=12, noop_seed=3)
    plain.reset()
    psnap = plain.save_state()
    assert psnap.rows == rec + 5
    before = (env.save_state().data.cpu().numpy(), env.stacked().cpu().numpy(), plain.save_state().data.cpu().numpy())
    with pytest.raises(_lib.ToyboxError):
        plain.load_state(snap)
    with pytest.raises(_lib.ToyboxError):
        env.load_state(psnap)
    after = (env.save_state().data.cpu().numpy(), env.stacked().cpu().numpy(), plain.save_state().data.cpu().numpy())
    assert all(np.array_equal(a, b) for a, b in zip(before, after))
    env.check()
    plain.check()
    env.close()
    plain.close()


def test_refusals():
    import torch
    from toybox_b200 import _lib
    from toybox_b200.wrappers import DeepmindToybox
    for p in (-0.01, 1.0000001, float("nan"), float("inf")):
        with pytest.raises(_lib.ToyboxError):
            DeepmindToybox("breakout", 4, repeat_action_probability=p)
    with pytest.raises(_lib.ToyboxError):
        DeepmindToybox("breakout", 4, max_episode_steps=-1)
    env = DeepmindToybox("breakout", 4)
    L, w = env.L, env._w
    trunc = torch.zeros(4, dtype=torch.uint8, device=env.device)
    assert L.tbx_wrap_set_sticky_actions(None, 0.5, 0) != 0 and L.tbx_wrap_set_time_limit(None, 10, None) != 0
    assert L.tbx_wrap_set_sticky_actions(w, -1.0, 0) != 0 and L.tbx_wrap_set_time_limit(w, -5, None) != 0
    assert L.tbx_wrap_set_sticky_actions(w, 0.5, 1) == 0 and L.tbx_wrap_state_rows(w) == L.tbx_state_rows(env.pool._h) + 7
    assert L.tbx_wrap_set_sticky_actions(w, 0.0, 1) == 0 and L.tbx_wrap_state_rows(w) == L.tbx_state_rows(env.pool._h) + 5
    assert L.tbx_wrap_set_time_limit(w, 0, C.c_void_p(trunc.data_ptr())) == 0
    env.reset()
    assert L.tbx_wrap_set_sticky_actions(w, 0.5, 1) != 0 and b"before the first" in L.tbx_last_error()
    assert L.tbx_wrap_set_time_limit(w, 10, None) != 0 and b"before the first" in L.tbx_last_error()
    assert L.tbx_wrap_state_rows(w) == L.tbx_state_rows(env.pool._h) + 5
    env.step(torch.zeros(4, dtype=torch.int32, device=env.device))
    env.check()
    env.close()
