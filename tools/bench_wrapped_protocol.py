"""Sticky actions and the episode time limit of the fused wrapper stack (DESIGN.md 4.5): time a wrapped agent step with each feature
against the default stack.  Per game, 65,536 envs at 84x84 (frame skip 4, max of two frames, FrameStack 4), six DeepmindToybox of the
same seeds stepping the same random action indices (generated on the device):

  off                   the defaults: the plain wrapper kernel + the dual gray tile kernel
  sticky                repeat_action_probability=0.25: the sticky wrapper kernel (one 64-bit mix per frame, two more words per env)
  sticky+limit          sticky and max_episode_steps=27000 (ALE v5's 108,000 frames at frame skip 4)
  <variant>/norender    step(render=False): the wrapper kernel alone

After --presteps untimed agent steps (steady state), the variants are timed in turn, --rounds rounds of --steps agent steps each (CUDA
events around each round), so that drift on a shared machine falls on all of them alike.  With p > 0 an env's trajectory differs from
the default one, so the sticky variants time other states than `off` (the line says so).  The GPU's name and power limit are read in the
same run.  --tree DIR imports toybox_b200 from another checkout (built in place) and times its default path only: run it before and
after a change, in one session, to compare the default path across versions.

    python tools/bench_wrapped_protocol.py [--envs 65536] [--presteps 200] [--rounds 5] [--steps 40] [--tree DIR] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAMES = ("breakout", "amidar", "space_invaders")
FEATURES = {"off": {}, "sticky": dict(repeat_action_probability=0.25),
            "sticky+limit": dict(repeat_action_probability=0.25, max_episode_steps=27000)}


def measure(DeepmindToybox, torch, game, n, presteps, rounds, steps, features):
    variants = [(f, r) for f in features for r in (True, False)]
    names = ["%s%s" % (f, "" if r else "/norender") for f, r in variants]
    envs = {name: DeepmindToybox(game, n, seeds=1, **FEATURES[f]) for name, (f, _) in zip(names, variants)}
    first = envs[names[0]]
    dev = first.device
    gen = torch.Generator(device=dev)
    gen.manual_seed(0xB200)
    acts = torch.randint(0, first.n_actions, (presteps + rounds * steps, n), generator=gen, device=dev, dtype=torch.int32)
    for name, (_, render) in zip(names, variants):
        e = envs[name]
        e.reset()
        for t in range(presteps):
            e.step(acts[t], render=render)
    torch.cuda.synchronize()
    ms = {v: [] for v in names}
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(rounds):
        t0 = presteps + r * steps
        for name, (_, render) in zip(names, variants):
            e = envs[name]
            start.record()
            for t in range(t0, t0 + steps):
                e.step(acts[t], render=render)
            stop.record()
            stop.synchronize()
            ms[name].append(start.elapsed_time(stop) / steps)
    trunc = {name: int(e.truncated.sum()) for name, e in envs.items() if hasattr(e, "truncated")}
    for e in envs.values():
        e.check()
        e.close()
    res = {"game": game, "size": "84x84", "envs": n, "presteps": presteps, "timed_agent_steps": rounds * steps}
    if len(features) > 1:
        res["states"] = "the sticky variants' trajectories diverge from off's: their rates are for other states"
    best = {v: min(ms[v]) for v in names}
    for v in names:
        res[v] = {"ms_per_agent_step": round(best[v], 4), "ms_rounds": [round(x, 4) for x in ms[v]],
                  "agent_steps_per_s": round(n / (best[v] * 1e-3))}
    for f in features:
        if f != "off" and "off" in features:
            res[f + "_over_off"] = round(best[f] / best["off"], 3)
            res[f + "_over_off_norender"] = round(best[f + "/norender"] / best["off/norender"], 3)
    if trunc:
        res["truncated_in_last_step"] = trunc
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--presteps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--games", default=",".join(GAMES))
    ap.add_argument("--tree", help="import toybox_b200 from this checkout and time its default path (variant off) only")
    ap.add_argument("--out", help="also append the lines to this file")
    args = ap.parse_args()
    tree = os.path.abspath(args.tree) if args.tree else ROOT
    sys.path.insert(0, tree)
    sys.path.insert(1, os.path.join(ROOT, "tools"))
    import torch
    import toybox_b200.wrappers as W                 # from `tree`: imported before anything else can import the package
    from bench_rgb_area import gpu_info
    if not torch.cuda.is_available():
        sys.exit("bench_wrapped_protocol.py needs a CUDA device")
    gpu = gpu_info(torch.cuda.current_device())
    features = ("off",) if args.tree else tuple(FEATURES)
    for game in args.games.split(","):
        res = measure(W.DeepmindToybox, torch, game, args.envs, args.presteps, args.rounds, args.steps, features)
        res.update({"tree": "--tree " + args.tree if args.tree else "this checkout", "gpu": gpu,
                    "timing": "CUDA events around each round of %d agent steps; the best round per variant, rounds alternating "
                              "the variants" % args.steps})
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
