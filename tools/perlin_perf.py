"""Cost of generating the reference's Perlin maps on the device (rtd3_perlin_maps) against the host's perlin_maps.

    python tools/perlin_perf.py [--reps 5] [--e2e-max 16384] [--out profiles/r6_perlin_maps.json]

Reports, in one run on one card:
  kernel   rtd3_perlin_maps alone for K = 1, 64, 1024, 16384, 65536 random seeds: CUDA events around back-to-back launches on
           preallocated buffers (about 0.2 s of launches per window), the median window of --reps with its spread.  The output
           (80 KB per map) is rewritten in place each launch, so for small K it stays in L2, as it does when rtd3_env_set_maps
           reads it next.
  tables   rtd3_env_set_maps on those maps (the table and halo build that set_perlin_maps adds), events as above.
  e2e      Environment.set_perlin_maps (4096 envs) for K up to --e2e-max: seed check, generation, table build and the one
           device-to-host copy of dynamics_speed / dynamics_angle, into a bank already allocated; host clock around the call
           and a device synchronise.
  host     environment.perlin_maps per map on this machine's CPU (the cache cleared), for three seeds.
The card's name, power limit and SM clock are read in the same run.
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

KS = (1, 64, 1024, 16384, 65536)


def time_launches(torch, fn, reps, window_s=0.2):
    """Median / min / max milliseconds per call of `fn` over `reps` windows of back-to-back calls."""
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    calls = int(min(1000, max(3, window_s / max(time.perf_counter() - t0, 1e-6))))
    per = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(calls):
            fn()
        b.record()
        b.synchronize()
        per.append(a.elapsed_time(b) / calls)
    return {"calls_per_window": calls, "ms_median": float(np.median(per)), "ms_min": min(per), "ms_max": max(per)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--e2e-max", type=int, default=16384, help="largest K timed end to end (its numpy copy is 80 KB per map)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_perlin_maps.json"))
    args = ap.parse_args()
    import torch
    import rtd3_b200 as rt
    from rtd3_b200 import environment as envmod

    if not torch.cuda.is_available():
        raise SystemExit("perlin_perf.py needs a GPU")
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
    lib = rt._lib
    L = lib.lib()
    W = rt.constants.WORLD_SIZE
    all_seeds = np.random.RandomState(0).randint(0, 2 ** 63, size=max(KS), dtype=np.int64)
    sampler = ClockSampler(0)
    sampler.start()
    sampler.in_region = True                                     # sampled over the whole device part
    t_start = time.time()

    env = rt.Environment(num_envs=4096, seed=0, map_seeds=all_seeds[:1])   # the first table build of each K allocates its bank
    kernel, tables = [], []
    for K in KS:
        seeds = torch.from_numpy(all_seeds[:K]).to(dev)
        speed = torch.empty((K, W, W), dtype=torch.float32, device=dev)
        angle = torch.empty_like(speed)
        gen = lambda: lib.check(L.rtd3_perlin_maps(lib.ptr(seeds), K, lib.ptr(speed), lib.ptr(angle), lib.stream_ptr(dev)), "perlin_maps")
        build = lambda: lib.check(L.rtd3_env_set_maps(env._handle, lib.ptr(speed), lib.ptr(angle), K, lib.stream_ptr(dev)), "env_set_maps")
        r = time_launches(torch, gen, args.reps)
        r.update(K=K, maps_per_s=K / (r["ms_median"] * 1e-3), us_per_map=r["ms_median"] * 1e3 / K)
        kernel.append(r)
        print("kernel  K=%6d  %9.3f ms  (%.2f us/map, spread %.3f-%.3f ms)" % (K, r["ms_median"], r["us_per_map"], r["ms_min"], r["ms_max"]),
              flush=True)
        r = time_launches(torch, build, args.reps)
        r.update(K=K)
        tables.append(r)
        print("tables  K=%6d  %9.3f ms" % (K, r["ms_median"]), flush=True)
        del seeds, speed, angle

    e2e = []
    for K in [k for k in KS if k <= args.e2e_max]:
        per = []
        for _ in range(max(3, args.reps // 2)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            env.set_perlin_maps(all_seeds[:K])
            torch.cuda.synchronize()
            per.append((time.perf_counter() - t0) * 1e3)
        e2e.append({"K": K, "ms_median": float(np.median(per)), "ms_min": min(per), "ms_max": max(per)})
        print("e2e     K=%6d  %9.3f ms" % (K, e2e[-1]["ms_median"]), flush=True)
    del env
    sampler.in_region = False
    sampler.stop()

    host = []
    for seed in (1707366464, 1, 2 ** 40 + 7):
        envmod._PERLIN_CACHE.pop(seed, None)
        t0 = time.perf_counter()
        envmod.perlin_maps(seed)
        host.append(time.perf_counter() - t0)
    print("host perlin_maps: %.3f s per map (median of %d seeds)" % (float(np.median(host)), len(host)), flush=True)

    out = {"card": card, "power_limit_w": power_w, "clocks": sampler.summary(), "reps": args.reps,
           "seconds": round(time.time() - t_start, 1), "kernel": kernel, "set_maps_tables": tables,
           "set_perlin_maps_e2e": {"num_envs": 4096, "rows": e2e},
           "host_perlin_maps_s_per_map": {"seeds": [1707366464, 1, 2 ** 40 + 7], "seconds": host, "median": float(np.median(host))}}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("# SM clock %s MHz (median over the device part); wrote %s" % (out["clocks"]["sm_mhz"], args.out), flush=True)


if __name__ == "__main__":
    main()
