"""Cost of the map bank (Environment maps=[K,100,100] + map_index) against the single-map kernels.

    python tools/map_bank_perf.py [--parts rollout,step,tick] [--reps 5] [--out-dir profiles]

Writes <out-dir>/r4_map_bank_{rollout,step,tick}.json.  Every configuration of one size runs on the same Environment (maps
switched with set_maps / set_map_index), and the configurations alternate within each repetition, so that clock drift
spreads over all of them; the median of the repetitions is kept, with the spread.  Timing: CUDA events around back-to-back
launches over rotating input buffers whose footprint exceeds the 126 MB L2 (as bench.py does).

  rollout  4096 x 1000, 65536 x 256, 1M x 64 steps: single map, K = 1 bank (index all 0), K = 8 / 64 / 512 contiguous blocks
           (512 maps over 4096 envs is 8 envs per map: every warp mixes maps), K = 128 in random warp-aligned blocks, K = 64
           per-env random.
  step     rtd3_env_step over 16.8M envs, single map (auto variant: the staged table) against K = 64 per-env random; bytes
           per env-step: 24 single map (state and action in, state out), 28 with a bank (+ the 4 B index entry).
  tick     BatchedTrainer fused tick, 8-tick graph, 8192 and 65536 envs, single map against K = 64 contiguous blocks; at 8192
           also the f16 multi-tick kernel (rtd3_tick_run_f16).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import ClockSampler  # noqa: E402

ROLL_SIZES = ((4096, 1000), (65536, 256), (1 << 20, 64))
STEP_N = 1 << 24


def maps_bank(rt, K):
    sp, an = zip(*[rt.synthetic_maps(k) for k in range(K)])
    return np.stack(sp), np.stack(an)


def configs(n, rs):
    """name -> (K, index or None); K = 0 is the single-map set_maps([100,100])."""
    warp_blocks = np.repeat(rs.randint(0, 128, (n + 31) // 32), 32)[:n]
    return {
        "single": (0, None),
        "bank_k1": (1, np.zeros(n, np.int32)),
        "k8_contiguous": (8, np.arange(n) * 8 // n),
        "k64_contiguous": (64, np.arange(n) * 64 // n),
        "k128_warp_aligned": (128, warp_blocks),
        "k512_contiguous": (512, np.arange(n) * 512 // n),
        "k64_per_env_random": (64, rs.randint(0, 64, n)),
    }


def apply(rt, env, bank, K, index):
    if K == 0:
        env.set_maps(*rt.synthetic_maps(0))
    else:
        env.set_maps(bank[0][:K], bank[1][:K], index=index)


def bench_rollout(rt, torch, dev, bank, reps, sampler, launches):
    L, sp, stream = rt._lib.lib(), rt._lib.stream_ptr(dev), torch.cuda.current_stream(dev)
    rows = []
    for n, T in ROLL_SIZES:
        env = rt.Environment(num_envs=n, seed=1707366464, maps=rt.synthetic_maps(0), device=dev)
        env.reset()
        start = env._state.clone()
        per_buf = T * 2 * n * 4
        R = max(2, int(np.ceil(160e6 / per_buf)) + 1)
        gen = torch.Generator(device=dev).manual_seed(T)
        acts = [torch.rand((T, 2, n), device=dev, generator=gen) * 15 - 7.5 for _ in range(R)]
        trajs = [torch.empty((T, 2, n), device=dev) for _ in range(R)]
        cfg = configs(n, np.random.RandomState(n))
        nl = max(4, int(launches * 4096 * 1000 / (n * T)))

        def go(k):
            q = k % R
            rt._lib.check(L.rtd3_env_rollout(env._handle, rt._lib.ptr(env._state[0]), rt._lib.ptr(env._state[1]),
                                             rt._lib.ptr(acts[q]), rt._lib.ptr(trajs[q]), n, T, sp))

        times = {name: [] for name in cfg}
        for r in range(reps + 1):                                # repetition 0 is the warm-up (and allocates the bank)
            for name, (K, index) in cfg.items():
                apply(rt, env, bank, K, index)
                env._state.copy_(start)
                for k in range(3):
                    go(k)
                torch.cuda.synchronize(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                sampler.in_region = True
                e0.record(stream)
                for k in range(nl):
                    go(k)
                e1.record(stream)
                torch.cuda.synchronize(dev)
                sampler.in_region = False
                if r:
                    times[name].append(e0.elapsed_time(e1) * 1e3 / nl)
        base = float(np.median(times["single"]))
        for name, (K, _) in cfg.items():
            us = float(np.median(times[name]))
            rows.append({"n": n, "T": T, "config": name, "K": K, "us_per_launch": round(us, 2),
                         "spread_us": round(max(times[name]) - min(times[name]), 2), "env_steps_per_sec": n * T / (us * 1e-6),
                         "vs_single": round(us / base, 3), "launches_per_window": nl})
            print("rollout %7d x %4d  %-20s %9.1f us  %.3e env-steps/s  x%.3f of single" % (n, T, name, us, n * T / (us * 1e-6), us / base),
                  flush=True)
        del env, acts, trajs
        torch.cuda.empty_cache()
    return rows


def bench_step(rt, torch, dev, bank, reps, sampler):
    L, sp, stream = rt._lib.lib(), rt._lib.stream_ptr(dev), torch.cuda.current_stream(dev)
    n = STEP_N
    env = rt.Environment(num_envs=4, seed=1, maps=rt.synthetic_maps(0), device=dev)   # the handle; the kernel takes any n
    bx = [torch.rand((2, n), device=dev) * 98 for _ in range(3)]                       # 3 rotating sets: > L2
    ba = [torch.rand((2, n), device=dev) * 15 - 7.5 for _ in range(3)]
    index = torch.from_numpy(np.random.RandomState(0).randint(0, 64, n).astype(np.int32)).to(dev)
    cfg = {"single": (24, 0), "k64_per_env_random": (28, 64)}
    times = {name: [] for name in cfg}

    def go(k):
        rt._lib.check(L.rtd3_env_step(env._handle, rt._lib.ptr(bx[k % 3][0]), rt._lib.ptr(bx[k % 3][1]),
                                      rt._lib.ptr(ba[k % 3][0]), rt._lib.ptr(ba[k % 3][1]), n, 0, sp))

    for r in range(reps + 1):
        for name, (_, K) in cfg.items():
            if K:
                env.set_maps(bank[0][:K], bank[1][:K], index=np.zeros(4, np.int32))
                rt._lib.check(L.rtd3_env_set_map_index(env._handle, rt._lib.ptr(index), n, sp))   # an index of n entries
            else:
                env.set_maps(*rt.synthetic_maps(0))
            for k in range(3):
                go(k)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sampler.in_region = True
            e0.record(stream)
            for k in range(30):
                go(k)
            e1.record(stream)
            torch.cuda.synchronize(dev)
            sampler.in_region = False
            if r:
                times[name].append(e0.elapsed_time(e1) * 1e3 / 30)
    rows = []
    for name, (bpe, K) in cfg.items():
        us = float(np.median(times[name]))
        gbs = n * bpe / (us * 1e-6) / 1e9
        rows.append({"n": n, "config": name, "K": K, "bytes_per_env_step": bpe, "us": round(us, 1),
                     "spread_us": round(max(times[name]) - min(times[name]), 1), "env_steps_per_sec": n / (us * 1e-6),
                     "GB/s": round(gbs, 1), "frac_of_7.7TB/s": round(gbs / 7700.0, 3)})
        print("step %d  %-20s %8.1f us  %.3e env-steps/s  %.0f GB/s at %d B" % (n, name, us, n / (us * 1e-6), gbs, bpe), flush=True)
    return rows


def bench_tick(rt, torch, dev, bank, reps, sampler):
    rows = []
    forms = (("fused, 8-tick graph", None, False), ("f16 8-tick kernel", "f16", True))
    for n in (8192, 65536):
        for label, precision, multi in forms:
            trainers = {}
            for name, K in (("single", 0), ("k64_contiguous", 64)):
                maps = rt.synthetic_maps(0) if K == 0 else (bank[0][:K], bank[1][:K])
                env = rt.Environment(num_envs=n, seed=1, maps=maps, device=dev)
                robot = rt.Robot(env.goal_state, hidden=256, layers=2, seed=100, buffer_size=max(50000, 16 * n))
                if precision:
                    robot.td3_agent.precision = precision
                robot.episodes_per_update = 10 ** 9
                robot.set_demonstration_states(np.random.RandomState(0).uniform(0, 99, (512, 2)))
                tr = rt.BatchedTrainer(env, robot, noise="philox", graph=True, check_interval=8, fused=True)
                tr.multi_tick_kernel = multi
                trainers[name] = tr
            if multi and not all(tr._multi_tick_ok() for tr in trainers.values()):
                continue                                         # the multi-tick kernel needs one wave of tiles (<= 18 944 envs)
            for tr in trainers.values():
                tr.run(32)
            torch.cuda.synchronize(dev)
            times = {name: [] for name in trainers}
            for r in range(reps):
                for name, tr in trainers.items():
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    sampler.in_region = True
                    e0.record()
                    tr.run(240)
                    e1.record()
                    torch.cuda.synchronize(dev)
                    sampler.in_region = False
                    times[name].append(e0.elapsed_time(e1) * 1e3 / 240)
            for name in trainers:
                us = float(np.median(times[name]))
                rows.append({"n": n, "form": label, "config": name, "us_per_tick": round(us, 2),
                             "spread_us": round(max(times[name]) - min(times[name]), 2), "env_steps_per_sec": n / (us * 1e-6)})
                print("tick %6d  %-20s %-16s %8.2f us/tick" % (n, label, name, us), flush=True)
            del trainers
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="rollout,step,tick")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--launches", type=int, default=32, help="rollout launches per timed window at 4096 x 1000 (scaled by size)")
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    import torch
    import rtd3_b200 as rt

    if not torch.cuda.is_available():
        raise SystemExit("map_bank_perf.py needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    card = torch.cuda.get_device_name(dev)
    power_w = None
    try:
        import pynvml
        pynvml.nvmlInit()
        power_w = pynvml.nvmlDeviceGetEnforcedPowerLimit(pynvml.nvmlDeviceGetHandleByIndex(0)) / 1000.0
    except Exception:
        pass
    print("# %s, power limit %s W" % (card, "%.0f" % power_w if power_w else "unknown"), flush=True)
    bank = maps_bank(rt, 512)
    os.makedirs(args.out_dir, exist_ok=True)
    parts = args.parts.split(",")
    for part, fn in (("rollout", lambda s: bench_rollout(rt, torch, dev, bank, args.reps, s, args.launches)),
                     ("step", lambda s: bench_step(rt, torch, dev, bank, args.reps, s)),
                     ("tick", lambda s: bench_tick(rt, torch, dev, bank, args.reps, s))):
        if part not in parts:
            continue
        sampler = ClockSampler(0)
        sampler.start()
        t0 = time.time()
        rows = fn(sampler)
        sampler.stop()
        out = {"card": card, "power_limit_w": power_w, "clocks": sampler.summary(), "reps": args.reps,
               "seconds": round(time.time() - t0, 1), "rows": rows}
        with open(os.path.join(args.out_dir, "r4_map_bank_%s.json" % part), "w") as f:
            json.dump(out, f, indent=1)
        print("# %s: SM clock %s MHz (median in the timed windows)" % (part, out["clocks"]["sm_mhz"]), flush=True)


if __name__ == "__main__":
    main()
