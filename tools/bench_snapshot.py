"""Device-resident state snapshots (DESIGN.md 4.7): time a full-pool save, a full-pool load and a 1 -> N fork, and the same
fork through the JSON codec.  Prints one JSON line per configuration: each game at 65,536 envs, and Breakout at a size whose
snapshot is larger than the B200's 126 MB L2.

Bytes are algorithmic: 4 * rows * k read plus 4 * rows * k written for a save or load, written only for a fork (one
column read).  The fraction is of the HBM peak bench.py uses (MEASURED_PEAKS.json hbm_gbs, else 6,650 GB/s).  Snapshots
that fit in L2 are read from it after the first launch; the last configuration does not fit.

    python tools/bench_snapshot.py [--iters 20] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import toybox_b200  # noqa: E402

CONFIGS = [("breakout", 65536), ("amidar", 65536), ("space_invaders", 65536), ("breakout", 524288)]


def hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback (bench.py)"


def gpu_info(index):
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["max_sm_clock_mhz"] = float(out[0]), float(out[1])
    except Exception as e:
        info["power_limit_w"] = "not read (%s)" % type(e).__name__
    return info


def timed(fn, iters):
    """ms per call: `iters` calls captured in one CUDA graph (a ~10 us copy would otherwise wait on the host), CUDA events
    around replays of it after a warm-up replay"""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(5):
        g.replay()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / (5 * iters)


def measure(game, n, iters, peak):
    pool = toybox_b200.BatchedToybox(game, n, seeds=1)
    for t in range(300):                              # mid-game states (content does not change the copy's cost)
        pool.step_random(7, t)
    L, h = pool.L, pool._h
    rows = L.tbx_state_rows(h)
    snap = pool.save_state()
    one = pool.save_state([0])
    buf = torch.empty_like(snap.data)
    zeros = torch.zeros(n, dtype=torch.int32, device=pool.device)
    blob = snap.tables
    stream = lambda: torch.cuda.current_stream().cuda_stream
    check = toybox_b200._lib.check
    copy_bytes = 4 * rows * n
    res = {"game": game, "envs": n, "rows": rows, "snapshot_mb": copy_bytes / 1e6}
    for name, fn, nbytes in (
            ("save", lambda: check(L.tbx_state_save(h, None, n, buf.data_ptr(), stream())), 2 * copy_bytes),
            ("load", lambda: check(L.tbx_state_load(h, snap.data.data_ptr(), n, None, None, n, blob, len(blob), stream())), 2 * copy_bytes),
            ("fork_1_to_n", lambda: check(L.tbx_state_load(h, one.data.data_ptr(), 1, zeros.data_ptr(), None, n, blob, len(blob), stream())),
             copy_bytes)):
        ms = timed(fn, iters)
        gbs = nbytes / (ms * 1e-3) / 1e9
        res[name] = {"ms": round(ms, 4), "bytes": nbytes, "gb_s": round(gbs, 1), "frac_of_peak": round(gbs / peak, 3)}
    pool.check()
    # the same 1 -> N fork through JSON: export env 0, import it into every env
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    doc = pool.to_state_json_text([0])[0]
    pool.write_state_json([doc] * n)
    torch.cuda.synchronize()
    res["fork_1_to_n_json_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
    res["fork_speedup_vs_json"] = round(res["fork_1_to_n_json_ms"] / res["fork_1_to_n"]["ms"], 1)
    pool.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", help="also append the lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_snapshot.py needs a CUDA device")
    peak, src = hbm_peak()
    gpu = gpu_info(torch.cuda.current_device())
    for game, n in CONFIGS:
        res = measure(game, n, args.iters, peak)
        res.update({"hbm_peak_gb_s": peak, "peak_source": src, "gpu": gpu, "timing": "CUDA events, 5 replays of a graph of %d calls" % args.iters})
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
