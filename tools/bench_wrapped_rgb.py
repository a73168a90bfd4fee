"""Colour observations of the fused wrapper stack (DeepmindToybox(grayscale=False), DESIGN.md 4.5 and 6): time a colour wrapped
agent step against a gray one on the same states.  Per game, 65,536 envs; three DeepmindToybox of the same seeds step the same
random action indices (generated on the device), so their states stay identical:

  gray       grayscale=True, 84x84 (frame skip 4, max of two frames, FrameStack 4): tbx_wrap_step + the dual gray tile kernel
  rgb        grayscale=False, 84x84: tbx_wrap_step + the dual RGB tile kernel
  norender   step(render=False): the wrapper kernel alone, so that gray - norender and rgb - norender are the renders' shares

After --presteps untimed agent steps (steady state), the variants are timed in turn, --rounds rounds of --steps agent steps each
(CUDA events around each round), so that drift on a shared machine falls on all three alike.  Breakout also runs at 64x64.
Bytes are algorithmic, per agent step: the render writes one observation (w * h * channels) and reads two state records per
env; the wrapper kernel reads and writes the record and writes the previous-state copy.  The GPU's name and power limit are read
in the same run.

    python tools/bench_wrapped_rgb.py [--envs 65536] [--presteps 300] [--rounds 4] [--steps 60] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from toybox_b200.wrappers import DeepmindToybox  # noqa: E402
from bench_rgb_area import gpu_info  # noqa: E402  (tools/ is on sys.path when this file runs)

CASES = (("breakout", (84, 84)), ("amidar", (84, 84)), ("space_invaders", (84, 84)), ("breakout", (64, 64)))
VARIANTS = ("gray", "rgb", "norender")


def measure(game, size, n, presteps, rounds, steps):
    envs = {"gray": DeepmindToybox(game, n, seeds=1, size=size), "rgb": DeepmindToybox(game, n, seeds=1, size=size, grayscale=False)}
    envs["norender"] = DeepmindToybox(game, n, seeds=1, size=size)
    n_act = envs["gray"].n_actions
    dev = envs["gray"].device
    gen = torch.Generator(device=dev)
    gen.manual_seed(0xB200)
    acts = torch.randint(0, n_act, (presteps + rounds * steps, n), generator=gen, device=dev, dtype=torch.int32)
    for name, e in envs.items():
        e.reset()
        for t in range(presteps):
            e.step(acts[t], render=name != "norender")
    torch.cuda.synchronize()
    ms = {v: [] for v in VARIANTS}
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(rounds):
        t0 = presteps + r * steps
        for name in VARIANTS:
            e = envs[name]
            start.record()
            for t in range(t0, t0 + steps):
                e.step(acts[t], render=name != "norender")
            stop.record()
            stop.synchronize()
            ms[name].append(start.elapsed_time(stop) / steps)
    same = torch.equal(envs["gray"].score, envs["rgb"].score) and torch.equal(envs["gray"].score, envs["norender"].score)
    rec = 4 * envs["gray"].pool.L.tbx_state_rows(envs["gray"].pool._h)
    for e in envs.values():
        e.check()
        e.close()
    w, h = size
    res = {"game": game, "size": "%dx%d" % size, "envs": n, "presteps": presteps, "timed_agent_steps": rounds * steps,
           "same_states": bool(same), "record_bytes": rec}
    best = {v: min(ms[v]) for v in VARIANTS}
    for v in VARIANTS:
        ch = 3 if v == "rgb" else 1
        nbytes = n * (3 * rec + (0 if v == "norender" else ch * w * h + 2 * rec))
        res[v] = {"ms_per_agent_step": round(best[v], 4), "ms_rounds": [round(x, 4) for x in ms[v]],
                  "agent_steps_per_s": round(n / (best[v] * 1e-3)), "algorithmic_bytes": nbytes,
                  "gb_s": round(nbytes / (best[v] * 1e-3) / 1e9, 1)}
    render = {v: best[v] - best["norender"] for v in ("gray", "rgb")}
    res["render_ms"] = {v: round(x, 4) for v, x in render.items()}
    res["rgb_over_gray_render"] = round(render["rgb"] / render["gray"], 2) if render["gray"] > 0 else None
    res["rgb_over_gray_step"] = round(best["rgb"] / best["gray"], 2)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--presteps", type=int, default=300)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--out", help="also append the lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_wrapped_rgb.py needs a CUDA device")
    gpu = gpu_info(torch.cuda.current_device())
    for game, size in CASES:
        res = measure(game, size, args.envs, args.presteps, args.rounds, args.steps)
        res.update({"gpu": gpu, "timing": "CUDA events around each round of %d agent steps; the best round per variant, rounds "
                                           "alternating the variants" % args.steps})
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
