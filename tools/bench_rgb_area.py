"""Colour INTER_AREA observations (TBX_OBS_RGB_AREA, DESIGN.md 4.3): time the RGB render against the gray renders of the same
states.  Per game, 65,536 envs in steady state (2,000 untimed step_random frames, as bench.py), then at 84x84 and 64x64:

  rgb_area    ('rgb_area', w, h): the tile kernel's RGB mode
  gray_tile   ('gray_area', w, h) with TBX_AREA_KERNEL=tile: the gray tile kernel alone, the RGB mode's like-for-like
  gray        ('gray_area', w, h) as rendered by default (the direct kernel where it covers the size, else the tile kernel)
  rgb_native  the native RGB frame (W x H x 3), what a caller resizes without this layout

Each is timed with CUDA events around `--launches` back-to-back renders after a warm-up.  Bytes are algorithmic:
N * (frame bytes + record bytes) per launch -- the frame written and the env's state record read; the fraction is of the HBM
peak bench.py uses (MEASURED_PEAKS.json hbm_gbs, else 6,650 GB/s).  The GPU's name and power limit are read in the same run.

    python tools/bench_rgb_area.py [--envs 65536] [--launches 200] [--out FILE]
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

GAMES = ("breakout", "amidar", "space_invaders")
SIZES = ((84, 84), (64, 64))


def hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback (bench.py)"


def gpu_info(index):
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["smi_name"], info["power_limit_w"] = out[0].strip(), float(out[1])
    except Exception as e:
        info["power_limit_w"] = "not read (%s)" % type(e).__name__
    return info


def timed(pool, out, obs, launches, env):
    """ms per render: CUDA events around `launches` renders into `out`, after 10 warm-up renders; `env` is set meanwhile"""
    saved = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        for _ in range(10):
            pool.render(out=out, obs=obs)
        torch.cuda.synchronize()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(launches):
            pool.render(out=out, obs=obs)
        stop.record()
        stop.synchronize()
        return start.elapsed_time(stop) / launches
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def measure(game, n, launches, peak):
    pool = toybox_b200.BatchedToybox(game, n, seeds=1)
    for t in range(2000):
        pool.step_random(0xB200, t)
    torch.cuda.synchronize()
    rec_bytes = 4 * pool.L.tbx_state_rows(pool._h)
    H, W = pool.height, pool.width
    res = {"game": game, "envs": n, "presteps": 2000, "record_bytes": rec_bytes, "sizes": {}}
    rgb = torch.empty((n, H, W, 3), dtype=torch.uint8, device=pool.device)
    ms = timed(pool, rgb, "rgb", launches, {})
    nbytes = n * (3 * W * H + rec_bytes)
    res["rgb_native"] = {"ms": round(ms, 4), "bytes": nbytes, "gb_s": round(nbytes / (ms * 1e-3) / 1e9, 1),
                         "frac_of_peak": round(nbytes / (ms * 1e-3) / 1e9 / peak, 3)}
    del rgb
    for w, h in SIZES:
        row = {}
        for name, mode, ch, env in (("rgb_area", "rgb_area", 3, {}), ("gray_tile", "gray_area", 1, {"TBX_AREA_KERNEL": "tile"}),
                                    ("gray", "gray_area", 1, {})):
            out = torch.empty((n, h, w, ch), dtype=torch.uint8, device=pool.device)
            ms = timed(pool, out, (mode, w, h), launches, env)
            nbytes = n * (ch * w * h + rec_bytes)
            gbs = nbytes / (ms * 1e-3) / 1e9
            row[name] = {"ms": round(ms, 4), "bytes": nbytes, "gb_s": round(gbs, 1), "frac_of_peak": round(gbs / peak, 3)}
        row["rgb_over_gray_tile"] = round(row["rgb_area"]["ms"] / row["gray_tile"]["ms"], 2)
        res["sizes"]["%dx%d" % (w, h)] = row
    pool.check()
    pool.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--out", help="also append the lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_rgb_area.py needs a CUDA device")
    peak, src = hbm_peak()
    gpu = gpu_info(torch.cuda.current_device())
    for game in GAMES:
        res = measure(game, args.envs, args.launches, peak)
        res.update({"hbm_peak_gb_s": peak, "peak_source": src, "gpu": gpu,
                    "timing": "CUDA events around %d back-to-back renders after 10 warm-up renders" % args.launches})
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
