"""CPU tier: the checker of the fused wrapper stack's final observations (final_obs_ref.FinalObsEnv) on seeded oracle runs.
The final stack is the FrameStack the reference held just before the VecEnv worker's reset; every MaxAndSkipEnv stop index
occurs; and a game that ends before the step's last frame shows stale buffer slots, not the frames it ended on."""
import numpy as np
import pytest

import final_obs_ref as F
from oracle import oracle as O
from oracle import wrappers as OW


def _rollout(game, n, steps, kw, edit=F.breakout_stagger, seed0=900):
    """(env, step, done, info, previous stacked obs, MaxAndSkipEnv's observation) of every done agent step"""
    refs = [F.FinalObsEnv(game, seed0 + i, env_id=i, noop_seed=5, **kw) for i in range(n)]
    prev = [r.reset() for r in refs]
    for i, r in enumerate(refs):
        js = r.base.b.state_json(0)
        edit(js, i)
        r.base.b.write_state_json(0, js)
    n_act = len(refs[0].base.legal)
    out = []
    for t in range(steps):
        for i, r in enumerate(refs):
            stacked, _, done, info = r.step(O.action_index(0xB200, i, t, n_act))
            if done:
                out.append((i, t, info, prev[i]))
            else:
                assert info["final"] is None
            prev[i] = stacked
    return refs, out


@pytest.mark.parametrize("kw", [dict(), dict(stack_reset="zero", frame_stack=2), dict(frame_skip=3, fire_reset=False, noop_max=0)])
def test_final_stack_is_the_pre_reset_frame_stack(kw):
    skip = kw.get("frame_skip", 4)
    refs, dones = _rollout("breakout", 12, 40, kw)
    assert len(dones) >= 12
    stops = set()
    for i, t, info, prev in dones:
        fin = info["final"]
        assert fin.shape == prev.shape
        # the k-1 newest frames before the step, then the frame of the step
        assert np.array_equal(fin[:-1], prev[1:]), (i, t)
        if info["real_done"]:
            stops.add(info["stop"])
        else:
            assert info["stop"] == skip - 1, (i, t)      # lost lives and truncations run the whole MaxAndSkipEnv step
    assert stops == set(range(skip)), stops


def test_final_frame_is_max_of_buffer_slots():
    """the last frame of the final stack is WarpFrame(max(_obs_buffer)) as the reference leaves it; where the game ended
    before frame skip-1 that max uses stale slots, and on some steps it differs from the max of the frames the game ended on"""
    refs, dones = _rollout("breakout", 12, 40, dict())
    stale = fresh = 0
    for i, t, info, prev in dones:
        fin, last2 = info["final"], info["last2"]
        ended_on = OW.warp(np.maximum.reduce(last2), 84, 84)
        if info["stop"] == 3:
            assert np.array_equal(fin[-1], ended_on), (i, t)
            fresh += 1
        elif not np.array_equal(fin[-1], ended_on):
            stale += 1
    assert fresh > 0 and stale > 0, (fresh, stale)


def _zero_buffer_edit(js, i):
    """a ball leaving the bottom of the screen away from the paddle, one life: the game ends on frame 0"""
    js.update(lives=1, is_dead=False, reset=False)
    js["balls"] = [{"position": {"x": 30.0, "y": 160.0}, "velocity": {"x": 0.0, "y": 3.0}}]
    js["paddle"]["position"]["x"] = 200.0


def test_unwritten_buffer_is_a_zero_frame():
    """without FireResetEnv and NoopResetEnv no MaxAndSkipEnv step precedes the first agent step, so a game that ends on its
    frame 0 leaves both buffer slots unwritten: the final frame is all zeros"""
    for kw in (dict(fire_reset=False, noop_max=0), dict(fire_reset=False, noop_max=0, stack_reset="zero", frame_skip=3)):
        refs, dones = _rollout("breakout", 2, 1, kw, edit=_zero_buffer_edit)
        assert len(dones) == 2
        for i, t, info, prev in dones:
            assert info["real_done"] and info["stop"] == 0
            assert not info["final"][-1].any() and np.array_equal(info["final"][:-1], prev[1:])


def test_abi_declares_the_setter():
    from toybox_b200 import _lib
    assert "tbx_wrap_set_final_observations" in _lib.SIGNATURES
