"""Breakout gray84 render alone (the direct kernel and its empty env-list tile launch), timed at two pool sizes to separate the
per-launch fixed cost (the persistent CTAs' prologue -- loading the shared-memory tables -- and tail) from the per-env cost.

  4,736 envs:  one 4-env chunk per team at 592 CTAs (148 SMs x 4 resident CTAs, 2 teams each): every team renders one chunk
  65,536 envs: the headline pool size

Each pool is brought to steady state first (2,000 untimed step_random frames, as bench.py), then `--launches` back-to-back
renders into one buffer are timed with CUDA events after 10 warm-up renders; the best of `--repeats` such windows is kept.
per_env_us = (t65536 - t4736) / (65,536 - 4,736), fixed_us = t4736 - 4,736 * per_env_us.  The GPU's name and power limit are
read in the same run.

    python tools/bench_direct_fixed.py [--launches 500] [--repeats 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import toybox_b200  # noqa: E402

SIZES = (4736, 65536)


def gpu_info(index):
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["smi_name"], info["power_limit_w"] = out[0].strip(), float(out[1])
    except Exception as e:
        info["power_limit_w"] = "not read (%s)" % type(e).__name__
    return info


def render_us(n, launches, repeats):
    pool = toybox_b200.BatchedToybox("breakout", n, seeds=1, obs="gray84")
    for t in range(2000):
        pool.step_random(0xB200, t)
    out = torch.empty((n,) + pool.obs_shape, dtype=torch.uint8, device=pool.device)
    for _ in range(10):
        pool.render(out=out)
    torch.cuda.synchronize()
    best = None
    for _ in range(repeats):
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(launches):
            pool.render(out=out)
        stop.record()
        stop.synchronize()
        us = start.elapsed_time(stop) * 1e3 / launches
        best = us if best is None else min(best, us)
    pool.check()
    pool.close()
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=500)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", help="also append the line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_direct_fixed.py needs a CUDA device")
    t = {n: render_us(n, args.launches, args.repeats) for n in SIZES}
    per_env = (t[SIZES[1]] - t[SIZES[0]]) / (SIZES[1] - SIZES[0])
    res = {"kernel": "brk_direct_kernel + empty env-list tile launch (Breakout gray84, steady state)",
           "render_us": {str(n): round(v, 2) for n, v in t.items()},
           "per_env_ns": round(per_env * 1e3, 4), "fixed_us": round(t[SIZES[0]] - SIZES[0] * per_env, 2),
           "gpu": gpu_info(torch.cuda.current_device()),
           "timing": "CUDA events around %d back-to-back renders after 10 warm-up renders, best of %d" % (args.launches, args.repeats)}
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
