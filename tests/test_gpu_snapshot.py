"""GPU tier: device-resident state snapshots (tbx_state_save / tbx_state_load, BatchedToybox.save_state / load_state / fork and
the wrapped-env forms): exact restore, forks against the oracle, partial / duplicate lists, foreign tables, invalid input,
CUDA-graph capture and checkpoints through torch.save."""
import copy
import io
import struct

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GAMES = ("breakout", "amidar", "space_invaders")
ORACLE_MODE = {"rgb": "rgb", "gray84": "gray84"}


@pytest.fixture(scope="module")
def tbx():
    import toybox_b200
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    toybox_b200.lib()
    return toybox_b200


@pytest.fixture(scope="module")
def oracle():
    from oracle import oracle as O
    O.lib()
    return O


def actions(O, game, n, t, seed):
    legal = np.asarray(O.LEGAL[game], np.int32)
    return legal[[O.action_index(seed, i, t, len(legal)) for i in range(n)]]


def steady_pool(tbx, game, n, seed, frames):
    """a pool whose envs have lost lives and restarted games"""
    pool = tbx.BatchedToybox(game, n, seeds=seed)
    for t in range(frames):
        pool.step_random(seed, t)
    return pool


def rollout(pool, seed, t0, frames, render_every=20):
    """per frame reward / done / score / lives, and gray84 + rgb frames every render_every frames"""
    out = []
    for t in range(t0, t0 + frames):
        pool.step_random(seed, t)
        out.append(torch.stack([pool.reward, pool.done.int(), pool.score, pool.lives]).cpu().numpy())
        if (t - t0) % render_every == render_every - 1:
            out.append(pool.render(obs="gray84").cpu().numpy())
            out.append(pool.render(obs="rgb").cpu().numpy())
    return out


def same(a, b):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert np.array_equal(x, y), i


def check_frames_vs_oracle(pool, ref, n):
    for mode in ("gray84", "rgb"):
        got = pool.render(obs=mode).cpu().numpy().reshape(n, -1)
        want = ref.render(ORACLE_MODE[mode]).reshape(n, -1)
        bad = np.argwhere(got != want)
        assert bad.size == 0, (mode, bad[:5])


@pytest.mark.parametrize("game", GAMES)
def test_save_step_load_replays_bit_identically(tbx, game):
    n, seed, K = 96, 11, 300
    pool = steady_pool(tbx, game, n, seed, frames=2000)
    assert pool.episode_stats()[0] > 0, "the pool should be in steady state (episodes ended)"
    snap = pool.save_state()
    assert snap.game == game and snap.rows == pool.L.tbx_state_rows(pool._h) and snap.k == n and not snap.wrapped
    first = rollout(pool, seed, 2000, K)
    assert sum(int(x[1].sum()) for x in first if x.ndim == 2 and x.shape[0] == 4) > 0, "episodes should end between save and load"
    js_first = pool.to_state_json_text()
    stats = pool.episode_stats()
    pool.load_state(snap)
    pool.check()
    assert pool.episode_stats() == stats          # pool-wide statistics are not env state
    second = rollout(pool, seed, 2000, K)
    same(first, second)
    assert pool.to_state_json_text() == js_first
    pool.close()


@pytest.mark.parametrize("game", GAMES)
def test_fork_matches_oracle_copy(tbx, oracle, game):
    n, seed = 32, 40
    pool = tbx.BatchedToybox(game, n, seeds=seed)
    ref = oracle.OracleBatch(game, n, seeds=seed + np.arange(n))
    for t in range(250):
        a = actions(oracle, game, n, t, 3)
        pool.apply_ale_action(a, auto_reset=True)
        ref.step(a, auto_reset=True)
    src = np.where(np.arange(n) % 3 == 0, 5, np.where(np.arange(n) % 3 == 1, 17, 26))   # every env, the sources included
    pool.fork(src)
    S, R = type(ref.states[0]), type(ref.sim[0])
    saved = {int(s): (S.from_buffer_copy(ref.states[s]), R.from_buffer_copy(ref.sim[s]), int(ref.prev_score[s])) for s in set(src)}
    for j, s in enumerate(src):
        st, sim, prev = saved[int(s)]
        ref.states[j] = S.from_buffer_copy(st)
        ref.sim[j] = R.from_buffer_copy(sim)
        ref.prev_score[j] = prev
    pool.check()
    for i in range(n):
        assert pool.to_state_json([i])[0] == ref.state_json(i), i
    check_frames_vs_oracle(pool, ref, n)
    for t in range(300):                          # each env its own action stream from here
        a = actions(oracle, game, n, t, 77)
        pool.apply_ale_action(a, auto_reset=True)
        r, d, s, l = ref.step(a, auto_reset=True)
        assert np.array_equal(pool.score.cpu().numpy(), s) and np.array_equal(pool.lives.cpu().numpy(), l), t
        assert np.array_equal(pool.reward.cpu().numpy(), r) and np.array_equal(pool.done.cpu().numpy().astype(bool), d), t
    for i in range(n):
        assert pool.to_state_json([i])[0] == ref.state_json(i), i
    check_frames_vs_oracle(pool, ref, n)
    pool.close()


@pytest.mark.parametrize("game", GAMES)
@pytest.mark.parametrize("on_device", [False, True])
def test_partial_and_duplicate_lists(tbx, game, on_device):
    n = 40
    a = steady_pool(tbx, game, n, 1, frames=300)
    b = steady_pool(tbx, game, n, 2, frames=200)
    src_ids = [1, 4, 7, 10, 4]
    dst_ids = [2, 5, 5, 9, 30]
    cols = [4, 0, 1, 2, 3]                        # entry j loads column cols[j]
    ids_in = lambda v: torch.tensor(v, dtype=torch.int32, device=a.device) if on_device else v
    snap = a.save_state(ids_in(src_ids))
    want_a = a.save_state().data.cpu().numpy()
    before = b.save_state().data.cpu().numpy()
    b.load_state(snap, env_ids=ids_in(dst_ids), columns=ids_in(cols))
    b.check()
    after = b.save_state().data.cpu().numpy()
    listed = set(dst_ids)
    for e in range(n):
        if e not in listed:
            assert np.array_equal(after[:, e], before[:, e]), e
    assert np.array_equal(after[:, 2], want_a[:, src_ids[cols[0]]])
    assert np.array_equal(after[:, 5], want_a[:, src_ids[cols[2]]])      # the last listed entry for env 5 wins, whole
    assert np.array_equal(after[:, 9], want_a[:, src_ids[cols[3]]])
    assert np.array_equal(after[:, 30], want_a[:, src_ids[cols[4]]])
    assert b.to_state_json([5])[0] == a.to_state_json([src_ids[cols[2]]])[0]
    a.close()
    b.close()


def _edited_states(game, states, rng):
    for i, js in enumerate(states):
        if game == "breakout":
            for k in rng.choice(108, size=int(rng.integers(0, 60)), replace=False):
                js["bricks"][int(k)]["alive"] = False
            if i % 2 == 0:
                js["bricks"][int(rng.integers(108))]["color"] = {"r": 250, "g": 250, "b": 250, "a": 255}
            if i % 3 == 0:
                js["bricks"][int(rng.integers(108))]["position"]["x"] += 3.0
        else:
            for _ in range(int(rng.integers(20, 120))):
                ty, tx = int(rng.integers(31)), int(rng.integers(32))
                js["board"]["tiles"][ty][tx] = ["Empty", "Unpainted", "ChaseMarker", "Painted"][int(rng.integers(4))]
            for b in js["board"]["boxes"]:
                b["painted"] = bool(rng.integers(2))
            if i % 2 == 0:                        # an edited box list: a table of its own
                box = js["board"]["boxes"][i % 5]
                box["triggers_chase"] = not box["triggers_chase"]
    return states


@pytest.mark.parametrize("game", ["breakout", "amidar"])
def test_foreign_tables_load_into_other_pools_and_configs(tbx, oracle, game):
    n = 24
    rng = np.random.default_rng(5)
    a = steady_pool(tbx, game, n, 8, frames=150)
    a.write_state_json(_edited_states(game, a.to_state_json(), rng))
    snap = a.save_state()
    assert snap.table_count > 1, "the edits should have added tables"
    want = a.to_state_json()
    other = a.config_to_json()
    if game == "breakout":
        other["row_colors"][0] = {"r": 10, "g": 200, "b": 30, "a": 255}
        other["paddle_color"] = {"r": 1, "g": 2, "b": 250, "a": 255}
    else:
        other["painted_color"] = {"r": 200, "g": 10, "b": 10, "a": 255}
        other["unpainted_color"] = {"r": 10, "g": 10, "b": 200, "a": 255}
    for cfg in (None, other):
        b = tbx.BatchedToybox(game, n, seeds=99, config=cfg)
        ref = oracle.OracleBatch(game, n, seeds=99 + np.arange(n), cfg_json=cfg)
        b.load_state(snap)
        b.check()
        got = b.to_state_json()
        for i in range(n):
            assert got[i] == want[i], i
            ref.write_state_json(i, want[i])
        check_frames_vs_oracle(b, ref, n)
        for t in range(60):
            acts = actions(oracle, game, n, t, 21)
            b.apply_ale_action(acts, auto_reset=True)
            ref.step(acts, auto_reset=True)
        check_frames_vs_oracle(b, ref, n)
        # a second load of the same snapshot finds its tables already interned
        b.load_state(snap)
        assert b.to_state_json() == want
        b.close()
    a.close()


@pytest.mark.parametrize("game", GAMES)
def test_invalid_entries_are_skipped_and_reported(tbx, tbx_error, game):
    n = 16
    a = steady_pool(tbx, game, n, 3, frames=120)
    b = steady_pool(tbx, game, n, 4, frames=60)
    snap = a.save_state()
    ref_a = snap.data.cpu().numpy()
    dev = a.device
    with pytest.raises(IndexError):
        b.load_state(snap, env_ids=[0, n])
    with pytest.raises(IndexError):
        a.save_state([-1])
    before = b.save_state().data.cpu().numpy()
    ids = torch.tensor([-1, 3, n + 50, 5, 6], dtype=torch.int32, device=dev)
    cols = torch.tensor([0, 1, 2, n + 7, 8], dtype=torch.int32, device=dev)
    bad_snap = copy.copy(snap)
    if game != "space_invaders":                  # env 6 would load a table index beyond the blob's tables
        bad_snap.data = snap.data.clone()
        bad_snap.data[14, 8] = snap.table_count + 3
    b.load_state(bad_snap, env_ids=ids, columns=cols)
    with pytest.raises(tbx_error, match="skipped"):
        b.check()
    b.check()                                     # reported once
    after = b.save_state().data.cpu().numpy()
    applied = {3: 1} if game != "space_invaders" else {3: 1, 6: 8}
    for e in range(n):
        assert np.array_equal(after[:, e], ref_a[:, applied[e]] if e in applied else before[:, e]), e
    a.save_state(torch.tensor([2, -4, n], dtype=torch.int32, device=dev))
    with pytest.raises(tbx_error, match="2 entries skipped"):
        a.check()
    # header mismatches are refused on the host before any device work
    for field, value in (("magic", 7), ("format", 99), ("game", (GAMES.index(game) + 1) % 3), ("rows", snap.rows + 1)):
        h = list(struct.unpack_from("<6I", snap.tables))
        h[["magic", "format", "game", "rows"].index(field)] = value
        forged = copy.copy(snap)
        forged.tables = struct.pack("<6I", *h) + snap.tables[24:]
        with pytest.raises(tbx_error):
            b.load_state(forged)
    other = tbx.BatchedToybox(GAMES[(GAMES.index(game) + 1) % 3], n, seeds=1)
    with pytest.raises(tbx_error):
        other.load_state(snap)
    other.close()
    assert np.array_equal(b.save_state().data.cpu().numpy(), after)
    b.check()
    a.close()
    b.close()


@pytest.fixture(scope="module")
def tbx_error(tbx):
    return tbx.ToyboxError


@pytest.mark.parametrize("game", GAMES)
def test_wrapped_env_save_load(tbx, game):
    from toybox_b200.wrappers import DeepmindToybox
    n, K = 24, 7                                  # K not a multiple of the stack depth: the ring head moves
    env = DeepmindToybox(game, n, seeds=12, noop_seed=3)
    env.reset()
    gen = np.random.default_rng(0)
    for _ in range(60):
        env.step(torch.as_tensor(gen.integers(0, env.n_actions, n), dtype=torch.int32, device=env.device))
    snap = env.save_state()
    assert snap.wrapped and snap.rows == tbx.lib().tbx_state_rows(env.pool._h) + 5
    stacked0 = env.stacked().cpu().numpy()
    acts = [torch.as_tensor(gen.integers(0, env.n_actions, n), dtype=torch.int32, device=env.device) for _ in range(K)]

    def run():
        out = []
        for a in acts:
            _, r, d, info = env.step(a)
            out += [env.stacked().cpu().numpy()] + [x.cpu().numpy().copy() for x in (r, d, info["real_done"], info["ep_return"], info["ep_length"])]
        return out

    first = run()
    env.load_state(snap)
    env.check()
    assert np.array_equal(env.stacked().cpu().numpy(), stacked0)
    same(first, run())
    # fork one env into every env: its ring and wrapper state follow
    env.fork([4])
    env.check()
    st = env.stacked().cpu().numpy()
    assert all(np.array_equal(st[i], st[4]) for i in range(n))
    with pytest.raises(ValueError):
        env.pool.load_state(snap)                 # a wrapped snapshot carries wrapper words
    env.close()


def test_cuda_graph_fork_step_render(tbx):
    n = 64
    pool = steady_pool(tbx, "breakout", n, 9, frames=200)
    dev = pool.device
    src = torch.tensor([5], dtype=torch.int32, device=dev)
    dst = torch.arange(n - 1, -1, -1, dtype=torch.int32, device=dev)       # a listed destination: the owner pass is captured too
    act = torch.zeros(n, dtype=torch.int32, device=dev)
    out = torch.empty((n,) + pool.obs_shape, dtype=torch.uint8, device=dev)
    legal = torch.tensor(pool.get_legal_action_set(), dtype=torch.int32, device=dev)

    def seq():
        pool.fork(src, dst)
        pool.apply_ale_action(act, auto_reset=True)
        pool.render(out=out)

    def record():
        return [x.cpu().numpy().copy() for x in (out, pool.reward, pool.done, pool.score, pool.lives)] + [pool.save_state().data.cpu().numpy()]

    start = pool.save_state()
    act.copy_(legal[torch.arange(n, device=dev) % len(legal)])
    seq()                                         # the first load allocates the owner array; the render path its lists
    torch.cuda.synchronize()
    pool.load_state(start)
    eager = []
    for _ in range(3):
        seq()
        eager += record()
    pool.load_state(start)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        seq()
    replay = []
    for _ in range(3):
        g.replay()
        replay += record()
    same(eager, replay)
    pool.check()
    pool.close()


@pytest.mark.parametrize("game", GAMES)
def test_checkpoint_round_trip(tbx, game):
    n, seed = 48, 6
    pool = steady_pool(tbx, game, n, seed, frames=300)
    buf = io.BytesIO()
    torch.save(pool.save_state(), buf)
    first = rollout(pool, seed, 300, 80)
    buf.seek(0)
    snap = torch.load(buf)
    fresh = tbx.BatchedToybox(game, n, seeds=1000)
    fresh.load_state(snap)
    same(first, rollout(fresh, seed, 300, 80))
    assert fresh.to_state_json_text() == pool.to_state_json_text()
    pool.close()
    fresh.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_checkpoint_across_devices(tbx):
    n, seed = 48, 6
    pool = steady_pool(tbx, "amidar", n, seed, frames=300)
    snap = pool.save_state()
    first = rollout(pool, seed, 300, 80)
    other = tbx.BatchedToybox("amidar", n, device="cuda:1", seeds=1000)
    other.load_state(snap)                        # copied to cuda:1 first
    same(first, rollout(other, seed, 300, 80))
    moved = snap.to("cuda:1")
    assert moved.device == torch.device("cuda", 1) and moved.game == "amidar"
    pool.close()
    other.close()
