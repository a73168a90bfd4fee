"""GPU tier: final observations of the fused wrapper stack (DeepmindToybox(final_observation=True),
tbx_wrap_set_final_observations) against the checker (final_obs_ref.FinalObsEnv), env by env and bit for bit, in the style
of test_gpu_wrapped_protocol._run: every step compares the stacked observation, reward, done, real done and truncation flag,
and where done the final stack.

Covered: the three games with real game overs, every MaxAndSkipEnv stop index; both stack modes and frame_stack 1 and 2;
frame_skip 1 and 3; a chain without FireResetEnv and NoopResetEnv; colour; sticky actions with a short time limit; a game
that ends before any buffer slot was written; unchanged outputs with the feature on and off; snapshots (same and other
config, corrupted carried records, refusals across wraps with and without the feature); CUDA-graph capture; render=False;
ToyboxVecEnv's terminal_observation; the setter's refusals."""
import ctypes as C

import numpy as np
import pytest

import final_obs_ref as F

pytestmark = pytest.mark.gpu
GAMES = ["breakout", "amidar", "space_invaders"]


def _acts(O, n, t, n_act):
    return np.asarray([O.action_index(0xB200, i, t, n_act) for i in range(n)], np.int32)


def _run(game, n, steps, kw, seed0=500, grayscale=True, edit=None):
    """returns (stop indices of the real game overs, number of done steps, number of truncations)"""
    import torch
    from oracle import oracle as O
    from toybox_b200.wrappers import DeepmindToybox
    env = DeepmindToybox(game, n, seeds=seed0, noop_seed=7, grayscale=grayscale, final_observation=True, **kw)
    refs = [F.FinalObsEnv(game, seed0 + i, env_id=i, noop_seed=7, **kw) for i in range(n)]
    if not grayscale:
        import wrapped_protocol_ref as R
        refs = [R.colour(r, kw.get("size", (84, 84))) for r in refs]
    obs = env.reset()
    assert np.array_equal(obs[:, env.order()].cpu().numpy(), np.stack([r.reset() for r in refs])), "reset"
    if edit is not None:
        states = []
        for i, r in enumerate(refs):
            js = r.base.b.state_json(0)
            edit(js, i)
            r.base.b.write_state_json(0, js)
            states.append(js)
        env.pool.write_state_json(states)
    stops, ndone, ntrunc = set(), 0, 0
    for t in range(steps):
        acts = _acts(O, n, t, env.n_actions)
        obs, rew, done, info = env.step(torch.as_tensor(acts, device=env.device))
        order = env.order()
        got = obs[:, order].cpu().numpy()
        fin = info["final_obs"][:, order].cpu().numpy()
        rew, done = rew.cpu().numpy(), done.cpu().numpy().astype(bool)
        real, trunc = info["real_done"].cpu().numpy().astype(bool), info["truncated"].cpu().numpy().astype(bool)
        for i, r in enumerate(refs):
            w_obs, w_rew, w_done, w_info = r.step(int(acts[i]))
            assert (w_rew, w_done, w_info["real_done"], w_info["truncated"]) == (rew[i], done[i], real[i], trunc[i]), (game, t, i)
            assert np.array_equal(got[i], w_obs), (game, t, i)
            if w_done:
                bad = np.argwhere(fin[i] != w_info["final"])
                assert bad.size == 0, (game, t, i, w_info["stop"], bad[:4])
                ndone += 1
                if w_info["real_done"]:
                    stops.add(w_info["stop"])
            ntrunc += int(w_info["truncated"])
    env.check()
    env.close()
    return stops, ndone, ntrunc


@pytest.mark.parametrize("game", GAMES)
def test_games(game):
    if game == "breakout":
        stops, nd, _ = _run(game, 12, 60, dict(), edit=F.breakout_stagger)
        assert stops == {0, 1, 2, 3}, stops
    else:
        stops, nd, _ = _run(game, 12, 150, dict(), edit=F.one_life)
        assert stops, "no game over"


@pytest.mark.parametrize("kw", [dict(stack_reset="zero"), dict(frame_stack=1), dict(frame_stack=2, stack_reset="zero"), dict(frame_stack=2)])
def test_stacks(kw):
    stops, _, _ = _run("breakout", 12, 40, kw, edit=F.breakout_stagger)
    assert stops == {0, 1, 2, 3}, stops


@pytest.mark.parametrize("kw", [dict(frame_skip=1), dict(frame_skip=3), dict(fire_reset=False, noop_max=0),
                                dict(frame_skip=3, fire_reset=False, noop_max=0, episode_life=False, stack_reset="zero")])
def test_wrapper_settings(kw):
    stops, _, _ = _run("breakout", 12, 60, kw, edit=F.breakout_stagger)
    assert stops == set(range(kw.get("frame_skip", 4))), stops


def test_other_games_with_settings():
    _run("space_invaders", 6, 80, dict(frame_skip=3, fire_reset=False, noop_max=0, frame_stack=2), edit=F.one_life)
    _run("amidar", 6, 80, dict(frame_skip=1, stack_reset="zero"), edit=F.one_life)


def test_colour():
    stops, _, _ = _run("breakout", 12, 40, dict(), grayscale=False, edit=F.breakout_stagger)
    assert stops == {0, 1, 2, 3}, stops


def test_sticky_and_time_limit():
    """many truncations: their final frame comes from a whole MaxAndSkipEnv step"""
    _, nd, nt = _run("breakout", 10, 120, dict(repeat_action_probability=0.25, max_episode_steps=13), edit=F.one_life)
    assert nt >= 20, nt


def _zero_buffer_edit(js, i):
    js.update(lives=1, is_dead=False, reset=False)
    js["balls"] = [{"position": {"x": 30.0, "y": 160.0}, "velocity": {"x": 0.0, "y": 3.0}}]
    js["paddle"]["position"]["x"] = 200.0


def test_zero_buffer():
    """no buffer slot written before a game that ends on frame 0 of the first agent step: a zero final frame, next to envs
    whose final frame is rendered"""
    import torch
    from toybox_b200.wrappers import DeepmindToybox
    for kw in (dict(fire_reset=False, noop_max=0), dict(fire_reset=False, noop_max=0, frame_skip=3, stack_reset="zero", frame_stack=2)):
        stops, nd, _ = _run("breakout", 4, 3, kw, edit=lambda js, i: _zero_buffer_edit(js, i) if i % 2 == 0 else F.breakout_stagger(js, i))
        assert 0 in stops
    env = DeepmindToybox("breakout", 4, seeds=3, fire_reset=False, noop_max=0, final_observation=True)
    env.reset()
    env.final_obs.fill_(7)
    ring = env.obs.clone()
    js = env.pool.to_state_json()
    for j in js:
        _zero_buffer_edit(j, 0)
    env.pool.write_state_json(js)
    _, _, done, info = env.step(torch.zeros(4, dtype=torch.int32, device=env.device))
    assert done.all() and info["real_done"].all()
    fin = env.final_obs.cpu().numpy()
    others = [s for s in range(4) if s != env.slot]
    assert not fin[:, env.slot].any() and np.array_equal(fin[:, others], ring[:, others].cpu().numpy())
    env.close()


def _collect(env, acts, render=True):
    out = []
    for a in acts:
        obs, r, d, info = env.step(a, render=render)
        out.append([x.cpu().numpy().copy() for x in (obs, r, d, info["real_done"], info["truncated"], info["ep_return"], info["ep_length"],
                                                      info["lives"], info["score"])])
    return out


@pytest.mark.parametrize("game", GAMES)
def test_outputs_unchanged(game):
    import torch
    from toybox_b200.wrappers import DeepmindToybox
    n = 32
    gen = np.random.default_rng(1)
    acts = None
    runs = []
    for fo in (False, True):
        env = DeepmindToybox(game, n, seeds=21, noop_seed=2, max_episode_steps=25, final_observation=fo)
        acts = acts or [torch.as_tensor(gen.integers(0, env.n_actions, n), dtype=torch.int32, device=env.device) for _ in range(80)]
        env.reset()
        runs.append(_collect(env, acts) + [[env.save_state().data[:env.L.tbx_state_rows(env.pool._h) + 5].cpu().numpy()]])
        env.close()
    a, b = runs
    assert all(np.array_equal(x, y) for sa, sb in zip(a, b) for x, y in zip(sa, sb))


@pytest.mark.parametrize("game", GAMES)
def test_snapshots(game):
    import torch
    from toybox_b200 import _lib
    from toybox_b200 import snapshot as S
    from toybox_b200.wrappers import DeepmindToybox
    n, K = 24, 60
    mk = lambda fo=True, **kw: DeepmindToybox(game, n, seeds=12, noop_seed=3, max_episode_steps=20, final_observation=fo, **kw)
    env = mk()
    rec = env.L.tbx_state_rows(env.pool._h)
    env.reset()
    gen = np.random.default_rng(0)
    for _ in range(30):
        env.step(torch.as_tensor(gen.integers(0, env.n_actions, n), dtype=torch.int32, device=env.device))
    snap = env.save_state()
    assert snap.rows == rec + 5 + 1 + 2 * rec
    acts = [torch.as_tensor(gen.integers(0, env.n_actions, n), dtype=torch.int32, device=env.device) for _ in range(K)]

    def run(e):
        out = []
        for a in acts:
            _, _, d, info = e.step(a)
            dn = d.cpu().numpy().astype(bool)
            out.append((dn, e.final_stacked().cpu().numpy()[dn]))        # FrameStack order: the rings' head slots differ
        return out

    first = run(env)
    assert sum(d.sum() for d, _ in first) > 0
    fresh = mk()
    fresh.load_state(snap)
    fresh.check()
    second = run(fresh)
    assert all(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) for a, b in zip(first, second))
    if game != "space_invaders":
        # through a pool of another config (its tables differ, so the carried records' tbl words are remapped) and back
        cfg = env.pool.config_to_json()
        if game == "breakout":
            cfg["row_colors"][0] = {"r": 10, "g": 200, "b": 30, "a": 255}
        else:
            cfg["painted_color"] = {"r": 200, "g": 10, "b": 10, "a": 255}
        other = mk(config=cfg)
        other.load_state(snap)
        other.check()
        back = mk()
        back.load_state(other.save_state())
        back.check()
        assert all(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) for a, b in zip(first, run(back)))
        other.close()
        back.close()
        # a carried record whose tbl word is out of range: the entry is skipped, reported, and the env keeps its state
        bad = S.StateSnapshot(snap.data.clone(), snap.tables, wrapped=True, obs=snap.obs.clone(), slot=snap.slot)
        bad.data[snap.rows - rec + S.TBL_WORD, 1] = 1 << 20
        keep = mk()
        keep.reset()
        before = (keep.save_state().data.cpu().numpy(), keep.obs.cpu().numpy())
        keep.load_state(bad, env_ids=[0, 1], columns=[0, 1])
        with pytest.raises(_lib.ToyboxError):
            keep.check()
        after = (keep.save_state().data.cpu().numpy(), keep.obs.cpu().numpy())
        assert np.array_equal(before[0][:, 1], after[0][:, 1]) and np.array_equal(before[1][1], after[1][1])
        assert not np.array_equal(before[0][:, 0], after[0][:, 0])
        keep.close()
    # wraps with and without the feature refuse each other's snapshots
    plain = mk(False)
    plain.reset()
    with pytest.raises(_lib.ToyboxError, match="final observations"):
        plain.load_state(snap)
    with pytest.raises(_lib.ToyboxError, match="final observations"):
        fresh.load_state(plain.save_state())
    fresh.check()
    for e in (env, fresh, plain):
        e.close()


def test_cuda_graph_and_no_render():
    import torch
    from toybox_b200.wrappers import DeepmindToybox
    n = 64
    gen = np.random.default_rng(4)
    # one frame per ring: a captured step always writes ring slot 0, as the eager one does
    mk = lambda: DeepmindToybox("breakout", n, seeds=5, max_episode_steps=9, frame_stack=1, final_observation=True)
    acts = [torch.as_tensor(gen.integers(0, 4, n), dtype=torch.int32, device="cuda") for _ in range(30)]
    eager, graphed = mk(), mk()
    for e in (eager, graphed):
        e.reset()
    static = torch.zeros(n, dtype=torch.int32, device="cuda")
    graphed.step(static)
    eager.step(static)             # the same first step, outside the graph (module loads, first allocations)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            graphed.step(static)
    ndone = 0
    for a in acts:
        static.copy_(a)
        g.replay()
        _, _, d, info = eager.step(a)
        torch.cuda.synchronize()
        dn = d.cpu().numpy().astype(bool)
        assert np.array_equal(dn, graphed.done.cpu().numpy().astype(bool))
        assert np.array_equal(eager.final_obs.cpu().numpy()[dn], graphed.final_obs.cpu().numpy()[dn])
        assert np.array_equal(eager.obs.cpu().numpy(), graphed.obs.cpu().numpy())
        ndone += int(dn.sum())
    assert ndone > 0
    # steps without rendering leave the final ring alone
    before = eager.final_obs.clone()
    nd = 0
    for a in acts:
        _, _, d, _ = eager.step(a, render=False)
        nd += int(d.sum())
    assert nd > 0 and torch.equal(before, eager.final_obs)
    eager.check()
    for e in (eager, graphed):
        e.close()


def test_vec_env_terminal_observation():
    from oracle import oracle as O
    from toybox_b200.wrappers import ToyboxVecEnv
    n, kw = 8, dict(max_episode_steps=15)
    venv = ToyboxVecEnv("breakout", n, seeds=40, noop_seed=9, final_observation=True, **kw)
    refs = [F.FinalObsEnv("breakout", 40 + i, env_id=i, noop_seed=9, stack_reset="zero", **kw) for i in range(n)]
    venv.reset()
    for r in refs:
        r.reset()
    nterm = 0
    for t in range(60):
        acts = _acts(O, n, t, 4)
        obs, rew, done, infos = venv.step(acts)
        for i, r in enumerate(refs):
            w_obs, _, w_done, w_info = r.step(int(acts[i]))
            assert w_done == done[i] and ("terminal_observation" in infos[i]) == bool(done[i]), (t, i)
            if w_done:
                term = infos[i]["terminal_observation"]
                assert term.shape == obs[i].shape and np.array_equal(term, w_info["final"].transpose(1, 2, 0)), (t, i)
                nterm += 1
    assert nterm > 0
    venv.close()


def test_setter_refusals():
    import torch
    from toybox_b200.wrappers import DeepmindToybox
    env = DeepmindToybox("breakout", 4)
    L, w = env.L, env._w
    ring = torch.zeros_like(env.obs)
    rec = L.tbx_state_rows(env.pool._h)
    assert L.tbx_wrap_set_final_observations(None, C.c_void_p(ring.data_ptr())) != 0
    assert L.tbx_wrap_set_final_observations(w, C.c_void_p(ring.data_ptr() + 1)) != 0 and b"aligned" in L.tbx_last_error()
    assert L.tbx_wrap_set_final_observations(w, C.c_void_p(ring.data_ptr())) == 0 and L.tbx_wrap_state_rows(w) == 3 * rec + 6
    assert L.tbx_wrap_set_final_observations(w, None) == 0 and L.tbx_wrap_state_rows(w) == rec + 5
    env.reset()
    assert L.tbx_wrap_set_final_observations(w, C.c_void_p(ring.data_ptr())) != 0 and b"before the first" in L.tbx_last_error()
    with pytest.raises(RuntimeError):
        env.final_stacked()
    env.step(torch.zeros(4, dtype=torch.int32, device=env.device))
    env.check()
    env.close()
