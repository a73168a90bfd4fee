#!/usr/bin/env python
"""bench.py -- the hot path's headline measurement (BASELINE.json: env-steps/s and rendered frames/s at
batch N; workload = configs[1]: Breakout, 65,536 envs per GPU, grayscale 84x84 observations, random actions).

One "step" = one pass of the hot path over the whole batch: generate the synthetic action stream on the
device, advance every env one frame (tbx_step), render every env (tbx_render).  Prints ONE JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--game G] [--envs E] [--obs gray84|gray|rgb|rgba]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...     (N > 1, one rank per GPU)
    python bench.py --impl reference ...    times the CPU restatement of the reference path (oracle/) on the host cores
    python bench.py --game amidar --envs 262144 --obs rgb          BASELINE configs[2]
    python bench.py --interventions         supplementary: BASELINE configs[3], Space Invaders 262,144 envs with JSON state interventions
    python bench.py --mixed 1048576 [--gpus N under torchrun]    supplementary: BASELINE configs[4], 1/3 of the envs per game,
                                            NCCL all-reduce of the episode statistics every 256 steps (inside the timed region)
    python bench.py --wrapped [--game G]    supplementary: the fused DeepMind wrapper stack (agent steps/s; 1 agent step = 4 frames)
    python bench.py --policy track --presteps 3000    supplementary: mid-game Breakout states (scripted ball-tracking policy)
    python bench.py --dump-outputs DIR      also write what the last timed step returned (a seeded sample) as DIR/*.npy, so that
                                            two builds can be compared output for output on the same seeded inputs

The pool is in steady state when the clock starts (--presteps 2000 untimed step-only frames, default); the line also carries the survey's
protocol (warm-up 100, 5 x 1,000 steps: best, mean, SEM), fresh-game / mid-game sub-records, the e2e leg with its own PCIe roofline
(raw and wrapped env), the collective's cost (N > 1) and, at 8 GPUs, the batch-1M north_star sub-record.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree as build() left it (it may be read-only)

GAME_DTYPE = {"breakout": "f64+u8", "amidar": "i32+u8", "space_invaders": "i32+u8"}
ACTION_SEED = 0xB200


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--game", default="breakout")
    ap.add_argument("--envs", type=int, default=65536, help="envs per GPU")
    ap.add_argument("--obs", default="gray84")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--policy", default="random", choices=["random", "track"],
                    help="random = the headline uniform stream; track = scripted Breakout ball tracking (breaks bricks)")
    ap.add_argument("--presteps", type=int, default=2000,
                    help="untimed step-only frames before the warm-up (default 2000: a steady-state pool whose episodes end and restart)")
    ap.add_argument("--no-protocol", action="store_true", help="skip the canonical-protocol repeats (warm-up 100, 5 x T steps)")
    ap.add_argument("--protocol-steps", type=int, default=1000, help="T of the canonical protocol (SURVEY 8d)")
    ap.add_argument("--no-states", dest="states", action="store_false", help="skip the fresh-game / mid-game sub-records")
    ap.add_argument("--interventions", action="store_true",
                    help="supplementary line: BASELINE configs[3] -- every 64 steps export the state JSON of 1,024 random envs, mutate, import")
    ap.add_argument("--mixed", type=int, default=0, metavar="TOTAL_ENVS",
                    help="supplementary line: BASELINE configs[4] -- TOTAL_ENVS (e.g. 1048576) split 1/3 per game and evenly over the GPUs, "
                         "gray84, NCCL all-reduce of the episode statistics every 256 steps")
    ap.add_argument("--wrapped", action="store_true",
                    help="supplementary line: the fused DeepMind wrapper stack (frame skip 4, max of 2 frames, 84x84, FrameStack 4)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last of the --steps timed steps returned (observations, reward, done, score, lives of a fixed "
                         "seeded sample of rank 0's envs, and the episode statistics) as DIR/<name>.npy, float32 / float64, <= 64 MB")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.mixed or args.wrapped or args.interventions):
        ap.error("--dump-outputs applies to the headline measurement only")
    return args


def obs_bytes(game, obs):
    w, h = {"breakout": (240, 160), "amidar": (160, 250), "space_invaders": (320, 210)}[game]
    return {"gray84": 84 * 84, "gray": w * h, "rgb": w * h * 3, "rgba": w * h * 4}[obs]


def workload_name(game, envs, obs):
    return "%s batched %d envs/GPU, %s obs, uniform random legal actions, auto-reset" % (game, envs, obs)


DUMP_BYTES = 48 << 20       # the dumped sample stays under 64 MB whatever --envs / --obs ask for


def sample_outputs(ro, stats_dev, env0):
    """Host copies of what the pool's last step returned, for a fixed seeded sample of its envs: the observations as float32,
    the per-env scalars and the episode statistics as float64 (every value is an integer, so both are exact)."""
    import numpy as np
    import torch
    n, fb = ro.n, ro.obs[0].numel()
    k = min(n, DUMP_BYTES // (4 * fb + 8 * 4))
    ids = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    idx = torch.from_numpy(ids).to(ro.obs.device)
    out = {"env_ids": (env0 + ids).astype(np.float64),
           "obs": ro.obs.index_select(0, idx).float().cpu().numpy(),
           "episode_stats": stats_dev.double().cpu().numpy()}
    for name in ("reward", "done", "score", "lives"):
        out[name] = getattr(ro.pool, name).index_select(0, idx).double().cpu().numpy()
    return out


def dump_outputs(outputs, path):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(path, name + ".npy"), a)


# --------------------------------------------------------------------------------------------- CPU arm
def cpu_rollout(game, obs, n_envs, steps, threads):
    """Oracle (CPU restatement of the reference's engine) on `threads` host threads; returns (env-steps/s, seconds)."""
    os.environ["OMP_NUM_THREADS"] = str(threads)
    import numpy as np
    from oracle import oracle as O
    batch = O.OracleBatch(game, n_envs, seeds=1234 + np.arange(n_envs))
    batch.rollout(2, 0, ACTION_SEED, 0, obs)               # touch everything once
    sec, _, _ = batch.rollout(steps, 2, ACTION_SEED, 0, obs)
    return n_envs * steps / sec, sec


def reference_arm(args):
    """--impl reference: ctoybox itself cannot be installed here (third-party Rust, no network, no rustc), so the
    reference arm is the CPU oracle -- the restated engine -- run with every host thread on the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(cores)
    import numpy as np
    from oracle import oracle as O
    n_sample = 256 * cores
    batch = O.OracleBatch(args.game, n_sample, seeds=1234 + np.arange(n_sample))
    t = 0
    for _ in range(max(args.warmup, 1)):
        batch.rollout(1, t, ACTION_SEED, 0, args.obs)
        t += 1
    t0 = time.perf_counter()
    for _ in range(args.steps):
        batch.rollout(1, t, ACTION_SEED, 0, args.obs)
        t += 1
    sec = time.perf_counter() - t0
    value = n_sample * args.steps / sec
    sample = "%d envs x 1 frame (step + %s render) per step on %d OpenMP threads" % (n_sample, args.obs, cores)
    line = {
        "impl": "reference", "metric": "env-steps/sec with rendered frames", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": GAME_DTYPE[args.game], "data": "synthetic",
        "config": {"workload": workload_name(args.game, args.envs, args.obs), "sample": sample},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "ctoybox==0.5.0 (Rust) is not installable here; this is oracle/ (C restatement) on all host threads",
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML in-process every 2 ms (nvidia_ml_py), or the
    nvidia-smi query of B200_PROFILING.md when NVML cannot be loaded."""
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.thread = index, [], False, None
        self.nvml, self.handle, self.max_mhz = None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].strip().isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _run_nvml(self):
        n = self.nvml
        bits = [(n.nvmlClocksThrottleReasonHwSlowdown, "hw_slowdown"), (n.nvmlClocksThrottleReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                (n.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_thermal_slowdown"), (n.nvmlClocksThrottleReasonSwPowerCap, "sw_power_cap")]
        while not self.stop_flag:
            try:
                mhz = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append([str(mhz), str(self.max_mhz), "0"] + ["Active" if r & b else "Not Active" for b, _ in bits])
            except Exception:
                pass
            time.sleep(0.002)

    def _run(self):
        if self.nvml is not None:
            return self._run_nvml()
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().splitlines()
                if out:
                    self.samples.append([x.strip() for x in out[0].split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def start(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=6)
        sm = sorted(int(float(s[0])) for s in self.samples if s and s[0].replace(".", "").isdigit())
        reasons = set()
        for s in self.samples:
            for k, name in enumerate(self.NAMES):
                if len(s) > 3 + k and s[3 + k].lower().startswith("active"):
                    reasons.add(name)
        mx = [int(float(s[1])) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(self.samples), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# --------------------------------------------------------------------------------------------- GPU arm
def wrapped_arm(args):
    """Supplementary measurement (SURVEY 8 f1): agent steps of the fused wrapper stack; 1 agent step = 4 game frames."""
    import numpy as np
    import torch
    import toybox_b200
    from toybox_b200.wrappers import DeepmindToybox
    toybox_b200.lib()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    n = args.envs
    env = DeepmindToybox(args.game, n, device=dev, seeds=(1234 + np.arange(n, dtype=np.int64)) & 0xFFFFFFFF)
    env.reset()
    acts = torch.empty(n, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(ACTION_SEED)
    pool_acts = torch.randint(0, env.n_actions, (64, n), device=dev, dtype=torch.int32, generator=gen)
    for t in range(max(args.warmup, 3)):
        env.step(pool_acts[t % 64])
    torch.cuda.synchronize(dev)
    K = args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for t in range(K):
        env.step(pool_acts[t % 64])
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    env.check()
    line = {"metric": "agent-steps/sec through the fused wrapper stack", "value": n * K / (ms * 1e-3), "unit": "agent-steps/s",
            "game_frames_per_sec": 4 * n * K / (ms * 1e-3), "n_gpus": 1, "steps": K, "warmup": max(args.warmup, 3), "ms_per_step": ms / K,
            "higher_is_better": True, "supplementary": True, "dtype": GAME_DTYPE[args.game], "data": "synthetic",
            "config": {"workload": "%s %d envs, frame skip 4 + max of 2 frames + 84x84 INTER_AREA + FrameStack 4 ring, uniform random actions" % (args.game, n)},
            "gpu_launches": 2 * K, "launches_per_step": ["wrap_step_kernel", "area_tile_kernel (dual)"],
            "episode_stats": env.pool.episode_stats()}
    print(json.dumps(line), flush=True)
    env.close()


def interventions_arm(args):
    """Supplementary measurement, BASELINE.json configs[3]: Space Invaders, 262,144 envs (--envs), gray84, random actions; every
    64 steps the state JSON of 1,024 random envs is exported, mutated (lives, ufo.appearance_counter, one shield pixel) and
    imported again -- the batched form of toybox/interventions/base.py:387-408.  Reports env-steps/s with and without the
    interventions, and the JSON throughput of both directions, for the dict-level API (what the reference's Intervention does)
    and for the text-level API (export text, edit only what changes)."""
    import numpy as np
    import torch
    import toybox_b200
    toybox_b200.lib()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    game = args.game if args.game != "breakout" else "space_invaders"
    n = args.envs if args.envs != 65536 else 262144
    pool = toybox_b200.BatchedToybox(game, n, device=dev, obs=args.obs, seeds=(1234 + np.arange(n, dtype=np.int64)) & 0xFFFFFFFF)
    obs = torch.empty((n,) + pool.obs_shape, dtype=torch.uint8, device=dev)
    acts = torch.empty(n, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev)
    rng = np.random.default_rng(7)
    t = [0]

    def step(render=True):
        pool.fill_random_actions(acts, ACTION_SEED, t[0], 0)
        pool.apply_ale_action(acts, auto_reset=True)
        if render:
            pool.render(out=obs)
        t[0] += 1

    def mutate(js):
        js["lives"] = 1 + int(rng.integers(5))
        if "ufo" in js:
            js["ufo"]["appearance_counter"] = int(rng.integers(1, 400))
            sh = js["shields"][int(rng.integers(3))]
            px = sh["data"][int(rng.integers(len(sh["data"])))]
            px[int(rng.integers(len(px)))] = {"r": 0, "g": 0, "b": 0, "a": 0}
        return js

    jstat = {"export_s": 0.0, "import_s": 0.0, "bytes": 0, "rounds": 0, "host_edit_s": 0.0}

    def intervene(text_level):
        ids = rng.choice(n, size=1024, replace=False).astype(np.int32)
        torch.cuda.synchronize(dev)          # the queued steps finish first: the export timer sees the codec, not the rollout
        t0 = time.perf_counter()
        docs = pool.to_state_json_text(ids)
        t1 = time.perf_counter()
        if text_level:      # decode / re-encode only every 8th document; the others go back as the text they came as
            docs = [json.dumps(mutate(json.loads(d))).encode() if i % 8 == 0 else d for i, d in enumerate(docs)]
        else:
            docs = [mutate(json.loads(d)) for d in docs]
        t2 = time.perf_counter()
        pool.write_state_json(docs, ids)
        t3 = time.perf_counter()
        jstat["export_s"] += t1 - t0
        jstat["host_edit_s"] += t2 - t1
        jstat["import_s"] += t3 - t2
        jstat["bytes"] += sum(len(d) if isinstance(d, bytes) else 0 for d in docs) if text_level else 0
        jstat["rounds"] += 1
        return sum(len(d) for d in docs) if text_level else None

    for _ in range(args.presteps):
        step(render=False)
    for _ in range(max(args.warmup, 3)):
        step()
    intervene(True)
    torch.cuda.synchronize(dev)
    K = max(args.steps, 128)

    def run(mode):
        for k in jstat:
            jstat[k] = 0
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for k in range(K):
            step()
            if mode is not None and k % 64 == 63:
                intervene(mode == "text")
        torch.cuda.synchronize(dev)
        return time.perf_counter() - t0, dict(jstat)

    sec_plain, _ = run(None)
    sec_dict, st_dict = run("dict")
    sec_text, st_text = run("text")
    doc_bytes = len(pool.to_state_json_text([0])[0])

    def jrec(sec, st):
        mb = 1024 * doc_bytes * st["rounds"] / 1e6
        return {"value": n * K / sec, "unit": "env-steps/s", "rounds": st["rounds"], "export_MBps": mb / st["export_s"] if st["export_s"] else None,
                "import_MBps": mb / st["import_s"] if st["import_s"] else None, "export_ms_per_round": 1e3 * st["export_s"] / max(st["rounds"], 1),
                "import_ms_per_round": 1e3 * st["import_s"] / max(st["rounds"], 1), "host_edit_ms_per_round": 1e3 * st["host_edit_s"] / max(st["rounds"], 1)}

    line = {"metric": "env-steps/sec with rendered frames and mid-rollout JSON state interventions", "value": n * K / sec_dict, "unit": "env-steps/s",
            "n_gpus": 1, "steps": K, "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * sec_dict / K, "higher_is_better": True, "supplementary": True,
            "dtype": GAME_DTYPE[game], "data": "synthetic", "timing": "host wall clock around K steps incl. the interventions (they synchronise)",
            "config": {"workload": "%s %d envs, %s obs, random legal actions, auto-reset; every 64 steps: to_state_json of 1,024 random envs, mutate lives / "
                                   "ufo.appearance_counter / one shield pixel, write_state_json" % (game, n, args.obs),
                       "presteps": args.presteps, "json_bytes_per_env": doc_bytes},
            "without_interventions": {"value": n * K / sec_plain, "unit": "env-steps/s"},
            "dict_level_api": jrec(sec_dict, st_dict), "text_level_api": jrec(sec_text, st_text),
            "gpu_launches": 3 * K, "episode_stats": pool.episode_stats()}
    print(json.dumps(line), flush=True)
    pool.close()


def mixed_arm(args):
    """Supplementary measurement, BASELINE.json configs[4]: the mixed-game sweep.  Every rank owns one pool per game
    (its shard of that game's env-id range, seeds from the global env id); a step = fill + step + render of all three
    pools; every 256 steps the per-game episode statistics are all-reduced (NCCL, device side, inside the timed region) --
    the path's only collective."""
    import numpy as np
    import torch
    import toybox_b200
    from toybox_b200 import distributed as D
    toybox_b200.lib()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    games = list(toybox_b200.GAMES)
    per_game = [args.mixed // 3, args.mixed // 3, args.mixed - 2 * (args.mixed // 3)]
    pools, bufs = [], []
    for game, total in zip(games, per_game):
        env0, n = D.shard(total, rank, world)
        pool = toybox_b200.BatchedToybox(game, n, device=dev, obs="gray84", seeds=D.global_seeds(1234, env0, n))
        pools.append((pool, env0, n))
        bufs.append((torch.empty((n,) + pool.obs_shape, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.int32, device=dev)))
    stream = torch.cuda.current_stream(dev)
    sdev = torch.zeros((3, 4), dtype=torch.int64, device=dev)
    n_reduces = [0]

    def reduce_all():
        for k, (pool, _, _) in enumerate(pools):
            pool.episode_stats_into(sdev[k])
        if dist is not None:
            mx = sdev[:, 3].clone()
            dist.all_reduce(sdev, op=dist.ReduceOp.SUM)
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            sdev[:, 3] = mx
        n_reduces[0] += 1

    def step(t, render=True):
        for (pool, env0, n), (obs, acts) in zip(pools, bufs):
            pool.fill_random_actions(acts, ACTION_SEED, t, env0)
            pool.apply_ale_action(acts, auto_reset=True)
            if render:
                pool.render(out=obs)
        if render and t % 256 == 255:
            reduce_all()

    t = 0
    for _ in range(args.presteps):          # steady state: episodes end and restart inside the run
        step(t, render=False)
        t += 1
    for _ in range(max(args.warmup, 3)):
        step(t)
        t += 1
    reduce_all()
    n_reduces[0] = 0

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    K = max(args.steps, 512)                # at least two statistics reduces inside the timed region
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(K):
        step(t)
        t += 1
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    for pool, _, _ in pools:
        pool.check()
    reduces_in_region = n_reduces[0]
    reduce_all()
    stats = [[int(v) for v in row] for row in sdev.cpu()]
    if dist is not None:
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    if rank == 0:
        line = {"metric": "env-steps/sec with rendered frames, mixed games", "value": args.mixed * K / (ms * 1e-3), "unit": "env-steps/s",
                "n_gpus": world, "steps": K, "warmup": max(args.warmup, 3), "ms_per_step": ms / K, "higher_is_better": True,
                "scaling": "strong", "supplementary": True, "dtype": "f64+i32+u8", "data": "synthetic",
                "config": {"workload": "mixed-game sweep: %d envs total = %s, split evenly over %d GPU(s), gray84 obs, random legal actions, "
                                       "auto-reset, NCCL all-reduce of per-game episode statistics every 256 steps"
                                       % (args.mixed, " + ".join("%d %s" % (n, g) for g, n in zip(games, per_game)), world),
                           "presteps": args.presteps},
                "gpu_launches": 9 * K, "collective": {"op": "all_reduce (SUM + MAX) of 3 x [episodes, sum_return, sum_length | max_return] int64",
                                                      "every_steps": 256, "inside_timed_region": reduces_in_region},
                "episode_stats": {g: s for g, s in zip(games, stats)}}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def _sem(xs):
    n = len(xs)
    m = sum(xs) / n
    if n < 2:
        return m, 0.0
    var = sum((x - m) ** 2 for x in xs) / (n - 1)
    return m, (var / n) ** 0.5


def main():
    args = parse()
    if args.impl == "reference":
        reference_arm(args)
        return
    if args.mixed:
        mixed_arm(args)
        return
    if args.wrapped:
        wrapped_arm(args)
        return
    if args.interventions:
        interventions_arm(args)
        return
    import numpy as np
    import torch
    import toybox_b200
    toybox_b200.lib()            # raises if the CUDA library is missing: no fallback
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    from toybox_b200 import distributed as D
    all_cpus = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa_cpus = D.bind_to_gpu_numa(local)          # pinned host buffers of the e2e leg land on the GPU's own NUMA node
    stream = torch.cuda.current_stream(dev)
    fb = obs_bytes(args.game, args.obs)
    rec_bytes = 4 * {"breakout": 72, "amidar": 366, "space_invaders": 392}[args.game]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if dist is None:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    class Rollout:
        """one pool + its buffers + the benchmark's step (fill actions, step, render)"""

        def __init__(self, n, policy="random"):
            self.n, self.policy, self.env0, self.t = n, policy, rank * n, 0
            self.pool = toybox_b200.BatchedToybox(args.game, n, device=dev, obs=args.obs,
                                                  seeds=(1234 + self.env0 + np.arange(n, dtype=np.int64)) & 0xFFFFFFFF)
            self.obs = torch.empty((n,) + self.pool.obs_shape, dtype=torch.uint8, device=dev)
            self.actions = torch.empty(n, dtype=torch.int32, device=dev)

        def fill(self):
            if self.policy == "track":
                self.pool.fill_policy_actions(self.actions, 1, self.t)
            else:
                self.pool.fill_random_actions(self.actions, ACTION_SEED, self.t, self.env0)

        def step(self, ev=None, render=True):
            if ev is not None:
                ev[0].record(stream)
            if self.policy == "track":
                self.fill()
                self.pool.apply_ale_action(self.actions, auto_reset=True)
            else:       # the uniform stream is generated inside the step kernel (tbx_step_random): one launch
                self.pool.step_random(ACTION_SEED, self.t, self.env0, auto_reset=True)
            if ev is not None:
                ev[1].record(stream)
            if render:
                self.pool.render(out=self.obs)
            if ev is not None:
                ev[2].record(stream)
            self.t += 1

        def presteps(self, k):           # advance the games without rendering (untimed)
            for _ in range(k):
                self.step(render=False)

        def timed(self, k, split=False):
            """k steps between two events on the launching stream; returns (ms, step_ms, render_ms)"""
            evs = {i: [torch.cuda.Event(enable_timing=True) for _ in range(3)] for i in range(0, k, 4)} if split else {}
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for i in range(k):
                self.step(evs.get(i))
            e1.record(stream)
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1)
            if not split:
                return ms, None, None
            return ms, sum(e[0].elapsed_time(e[1]) for e in evs.values()) / len(evs), sum(e[1].elapsed_time(e[2]) for e in evs.values()) / len(evs)

        def close(self):
            self.pool.close()

    n = args.envs
    ro = Rollout(n, args.policy)
    pool = ro.pool
    ro.presteps(args.presteps)
    W = max(args.warmup, 3)
    for _ in range(W):
        ro.step()
    torch.cuda.synchronize(dev)

    # ---- the path's one collective, device side: the episode-statistics vector, summed / maxed over the GPUs by NCCL.  It
    # runs INSIDE the timed region (once, after the K-th step) and is timed on its own below.
    stats_dev = torch.zeros(4, dtype=torch.int64, device=dev)

    def reduce_stats():
        pool.episode_stats_into(stats_dev)
        if dist is not None:
            mx = stats_dev[3:].clone()
            dist.all_reduce(stats_dev, op=dist.ReduceOp.SUM)
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            stats_dev[3:] = mx

    reduce_stats()
    # ---- timed region: exactly K steps (+ the statistics reduce), device-timed, max over ranks
    K = args.steps
    # per-kernel events on every EV_STRIDE-th step of the region: an event between two launches serialises them (the next kernel's
    # first CTAs otherwise start while the previous kernel's tail drains, ~7 us per step here), so timing every launch would slow
    # the region it measures by 6 %
    EV_STRIDE = 4
    evs = {k: [torch.cuda.Event(enable_timing=True) for _ in range(3)] for k in range(0, K, EV_STRIDE)}
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    if dist is not None:        # device-side rendezvous: the ranks' streams pass this point together, whatever the skew of their host threads
        dist.all_reduce(torch.zeros(1, dtype=torch.int32, device=dev))
    e_start, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_start.record(stream)
    for k in range(K):
        ro.step(evs.get(k))
    reduce_stats()
    e_end.record(stream)
    barrier()
    ms = max_over_ranks(e_start.elapsed_time(e_end))
    step_ms = sum(e[0].elapsed_time(e[1]) for e in evs.values()) / len(evs)
    render_ms = sum(e[1].elapsed_time(e[2]) for e in evs.values()) / len(evs)
    pool.check()
    value = world * n * K / (ms * 1e-3)
    stats = [int(v) for v in stats_dev.cpu()]
    # copied now: the protocol repeats and the e2e leg below advance the same pool
    outputs = sample_outputs(ro, stats_dev, ro.env0) if args.dump_outputs and rank == 0 else None

    # ---- the survey's protocol (SURVEY 8d, after test/benchmark.py:119-166): warm-up 100, T = 1,000 timed steps, best of 5 and
    # mean +- SEM over the 5 repeats -- measured in the same run, after the driver's K-step region above
    protocol = None
    if not args.no_protocol:
        T, reps = args.protocol_steps, 5
        for _ in range(100):
            ro.step()
        vals = []
        for _ in range(reps):
            barrier()
            pms = max_over_ranks(ro.timed(T)[0])
            vals.append(world * n * T / (pms * 1e-3))
        mean, sem = _sem(vals)
        protocol = {"warmup": 100, "steps": T, "repeats": reps, "best": max(vals), "mean": mean, "sem": sem, "unit": "env-steps/s",
                    "note": "canonical protocol of SURVEY 8d; `value` above is the driver's --steps/--warmup region"}
    clocks = sampler.stop() if rank == 0 else None

    # ---- the collective on its own: 20 statistics reduces back to back
    collective = None
    if dist is not None:
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream)
        for _ in range(20):
            reduce_stats()
        c1.record(stream)
        barrier()
        collective = {"op": "NCCL all_reduce of [episodes, sum_return, sum_length | max_return] int64", "us": max_over_ranks(c0.elapsed_time(c1)) * 1e3 / 20,
                      "inside_timed_region": True}

    # ---- e2e: the same metric through the host-facing call (host actions in, host observations out), with its own
    # roofline: a bare pinned device->host copy of the same bytes, timed on every rank at the same time
    e2e = None
    if not args.no_e2e:
        rng = np.random.default_rng(rank)
        legal = np.asarray(pool.get_legal_action_set(), np.int32)
        h_actions = torch.from_numpy(legal[rng.integers(0, len(legal), size=n)]).pin_memory()
        h_obs = torch.empty((n,) + pool.obs_shape, dtype=torch.uint8).pin_memory()
        ke = max(3, min(K, 20))
        for _ in range(3):
            pool.step_host(h_actions, obs_out=h_obs)
        barrier()
        t0 = time.perf_counter()
        for _ in range(ke):
            pool.step_host(h_actions, obs_out=h_obs)
        barrier()
        sec = max_over_ranks(time.perf_counter() - t0)
        d2h = n * (fb + 4 + 1 + 4 + 4)
        for _ in range(2):
            h_obs.copy_(ro.obs, non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(ke):
            h_obs.copy_(ro.obs, non_blocking=True)
            torch.cuda.synchronize(dev)
        barrier()
        csec = max_over_ranks(time.perf_counter() - t0)
        pcie = n * fb * ke / csec / 1e9
        e2e = {"value": world * n * ke / sec, "unit": "env-steps/s", "h2d_bytes_per_step": 4 * n, "d2h_bytes_per_step": d2h, "steps": ke,
               "api": "BatchedToybox.step_host -> tbx_step_host (pinned host actions in; obs, reward, done, score, lives out)",
               "pcie_gbs": pcie, "achieved_gbs": d2h * ke / sec / 1e9, "frac": (d2h * ke / sec / 1e9) / pcie,
               "numa_bound_cpus": len(numa_cpus) if numa_cpus else None,
               "pcie_note": "pcie_gbs = a bare pinned cudaMemcpyAsync D2H of the observation bytes per rank, all %d rank(s) copying at the "
                            "same time: the host-side ceiling of this call" % world}
        del h_obs
        # the call a trainer makes: the wrapped env (frame skip 4 + max of 2 + 84x84 + 4-frame stack), host actions in, the observation
        # stack + reward + done out to pinned host memory -- one observation per 4 game frames
        if args.game == "breakout" and args.obs == "gray84":
            from toybox_b200.wrappers import DeepmindToybox
            wenv = DeepmindToybox(args.game, n, device=dev, seeds=(1234 + rank * n + np.arange(n, dtype=np.int64)) & 0xFFFFFFFF, env0=rank * n, stack_reset="zero")
            wenv.reset()
            hw_act = torch.from_numpy(rng.integers(0, wenv.n_actions, size=n).astype(np.int32)).pin_memory()
            d_act = torch.empty(n, dtype=torch.int32, device=dev)
            hw_obs = torch.empty((n, wenv.k, wenv.out_h, wenv.out_w), dtype=torch.uint8).pin_memory()
            hw_new = torch.empty((n, wenv.out_h, wenv.out_w), dtype=torch.uint8).pin_memory()
            d_new = torch.empty((n, wenv.out_h, wenv.out_w), dtype=torch.uint8, device=dev)
            hw_rew = torch.empty(n, dtype=torch.int32).pin_memory()
            hw_done = torch.empty(n, dtype=torch.uint8).pin_memory()

            def wstep(full):
                d_act.copy_(hw_act, non_blocking=True)
                wenv.step(d_act)
                if full:
                    hw_obs.copy_(wenv.obs, non_blocking=True)
                else:                   # the newest observation only (the host keeps the stack): gathered on the device, one contiguous copy
                    d_new.copy_(wenv.obs[:, wenv.slot])
                    hw_new.copy_(d_new, non_blocking=True)
                hw_rew.copy_(wenv.reward, non_blocking=True)
                hw_done.copy_(wenv.done, non_blocking=True)
                torch.cuda.synchronize(dev)

            wrapped = {}
            for name, full in (("stack_of_4", True), ("newest_frame", False)):
                for _ in range(3):
                    wstep(full)
                barrier()
                t0 = time.perf_counter()
                for _ in range(ke):
                    wstep(full)
                barrier()
                wsec = max_over_ranks(time.perf_counter() - t0)
                wb = n * (fb * (wenv.k if full else 1) + 4 + 1)
                wrapped[name] = {"agent_steps_per_sec": world * n * ke / wsec, "game_frames_per_sec": 4 * world * n * ke / wsec, "d2h_bytes_per_step": wb,
                                 "achieved_gbs": wb * ke / wsec / 1e9, "frac_of_pcie": (wb * ke / wsec / 1e9) / pcie}
            e2e["wrapped"] = wrapped
            e2e["wrapped_api"] = "DeepmindToybox.step (tbx_wrap_step): pinned host actions in; observation ring (or its newest slot), reward, done out to pinned host memory"
            wenv.close()
            del hw_obs, hw_new

    # ---- the same pool from other game states, as named sub-records (the render cost follows what differs from a fresh game)
    states = {}
    if args.states and args.game == "breakout" and args.obs == "gray84":
        def sub(name, policy, pre):
            r2 = Rollout(n, policy)
            r2.presteps(pre)
            for _ in range(5):
                r2.step()
            torch.cuda.synchronize(dev)
            barrier()
            sms, s_ms, r_ms = r2.timed(50, split=True)
            sms = max_over_ranks(sms)
            est = r2.pool.episode_stats()
            r2.close()
            states[name] = {"value": world * n * 50 / (sms * 1e-3), "unit": "env-steps/s", "steps": 50, "policy": policy, "presteps": pre,
                            "render_ms": r_ms, "step_ms": s_ms, "episodes": est[0]}
        sub("fresh_game", "random", 0)
        sub("midgame_tracking_policy_3000", "track", 3000)

    # ---- north_star: Breakout gray84 at batch 1M over 8 GPUs = 131,072 envs per GPU (the weak-scaling line above keeps --envs)
    north_star = None
    if world == 8 and args.game == "breakout" and args.obs == "gray84" and args.policy == "random":
        ro.close()
        r3 = Rollout(131072, "random")
        r3.presteps(args.presteps)
        for _ in range(W):
            r3.step()
        barrier()
        nms = max_over_ranks(r3.timed(max(K, 50))[0])
        north_star = {"value": world * 131072 * max(K, 50) / (nms * 1e-3), "unit": "env-steps/s", "total_envs": world * 131072,
                      "envs_per_gpu": 131072, "steps": max(K, 50), "presteps": args.presteps, "target": 1e9}
        ro = r3
        pool = ro.pool

    # ---- the HBM-bound layout of the same render path (native RGBA frames), same pool and states: supplementary roofline
    native = None
    if rank == 0 and args.obs == "gray84" and north_star is None:
        nb = obs_bytes(args.game, "rgba")
        if n * nb <= (24 << 30):
            big = torch.empty((n, nb), dtype=torch.uint8, device=dev)
            for _ in range(3):
                pool.render(out=big, obs="rgba")
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            torch.cuda.synchronize(dev)
            ev[0].record(stream)
            for _ in range(10):
                pool.render(out=big, obs="rgba")
            ev[1].record(stream)
            torch.cuda.synchronize(dev)
            nms = ev[0].elapsed_time(ev[1]) / 10
            nbytes = n * (nb + rec_bytes)
            native = {"kernel": "base_fill_kernel + native_patch_kernel<%s,rgba>" % args.game, "launch_ms": nms, "bytes_per_launch": nbytes,
                      "achieved": nbytes / (nms * 1e-3) / 1e9, "unit": "GB/s", "frames_per_sec": n / (nms * 1e-3)}
            del big
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (render): algorithmic bytes per launch / measured launch time
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak, peak_src = float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    alg_bytes = n * (fb + rec_bytes)          # frame written + state record read, per env, per launch
    achieved = alg_bytes / (render_ms * 1e-3) / 1e9
    if args.obs == "gray84":
        kname = "brk_direct_kernel" if args.game == "breakout" and os.environ.get("TBX_AREA_KERNEL") not in ("tile", "cta") else "area_tile_kernel<%s>" % args.game
    else:
        kname = "base_fill_kernel + native_patch_kernel<%s,%s>" % (args.game, args.obs)
    # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel on this workload, from the committed
    # `ncu --set full` capture (profiles/r2_traffic.json, written by tools/ncu_traffic.py); null when never captured
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        key = "%s/%s/%d" % (args.game, args.obs, n)
        if key in tr:
            traffic = tr[key]["dram_bytes"]
    except Exception:
        pass
    roofline = {"kernel": kname, "bound": "hbm", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "bytes_per_launch": alg_bytes, "launch_ms": render_ms, "step_kernel_ms": step_ms,
                "launch_ms_from": "CUDA events around every %d-th step's launches inside the timed region (%d samples)" % (EV_STRIDE, len(evs)),
                "note": "a 7 KB gray84 frame costs more instruction issue than DRAM time; the HBM-bound layout is in roofline.native"}
    if native is not None:
        native["frac"] = native["achieved"] / peak
    roofline["native"] = native
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        if all_cpus:
            os.sched_setaffinity(0, all_cpus)       # the CPU baseline uses every host core again
        cores = os.cpu_count() or 1
        n_cpu = 64 * cores
        v1, s1 = cpu_rollout(args.game, args.obs, n_cpu, 20, cores)
        steps_cpu = int(max(20, min(4000, 12.0 / (s1 / 20))))
        v, s = cpu_rollout(args.game, args.obs, n_cpu, steps_cpu, cores)
        cpu = {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port",
               "sample": "%d envs x %d frames (step + %s render), %.1f s, oracle/ C restatement with OpenMP" % (n_cpu, steps_cpu, args.obs, s)}
    launches = (["step_kernel (synthetic action stream fused)"] if args.policy == "random" else ["breakout_tracking_actions_kernel", "step_kernel"]) + [kname] + (["area_tile_kernel (env-list mode, normally empty)"] if kname == "brk_direct_kernel" else [])
    line = {
        "metric": "env-steps/sec with rendered frames", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": GAME_DTYPE[args.game], "data": "synthetic",
        "config": {"workload": workload_name(args.game, n, args.obs), "envs_per_gpu": n, "obs_bytes_per_env": fb,
                   "l2": "each step writes %d MB of observations (> 126 MB L2) between reuses of the %d MB state" %
                         (n * fb // 2 ** 20, n * rec_bytes // 2 ** 20),
                   "seeds": "env i: set_seed(1234+i); actions: counter-based stream seed 0xB200",
                   "policy": args.policy, "presteps": args.presteps,
                   "state": "steady state: %d untimed step-only frames before the warm-up, episodes end and auto-reset inside the run" % args.presteps},
        "frames_per_sec": value, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": len(launches) * K,
        "launches_per_step": launches, "protocol": protocol, "states": states or None, "collective": collective, "north_star_1M": north_star,
        "clocks": clocks, "episode_stats": {"episodes": stats[0], "sum_return": stats[1], "sum_length": stats[2], "max_return": stats[3],
                                            "scope": "all ranks (NCCL-reduced), since pool creation"},
    }
    if outputs is not None:
        dump_outputs(outputs, args.dump_outputs)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
