"""Per-step cost and fixed cost of rtd3_env_rollout: time = a + b*T, fitted over T at each batch size.

    python tools/rollout_slope.py [--n 1024,4096,8192] [--T 125,250,500,1000,2000] [--launches 64] [--reps 3] [--json FILE]

Each point is `launches` back-to-back launches timed with CUDA events, over rotating action / trajectory buffers whose
footprint exceeds the 126 MB L2 (as bench.py does); the median of `reps` windows is kept.  b is printed in ns and in SM
cycles per step at the median SM clock NVML reported during the windows, a as the fixed cost of one launch.  The headline
(bench.py) cannot separate the two: a change to the per-step chain shows in b, a change to launch / staging cost in a.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import ClockSampler  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", default="1024,4096,8192")
    ap.add_argument("--T", default="125,250,500,1000,2000")
    ap.add_argument("--launches", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--json", default=None, help="also write the points and fits to this file")
    args = ap.parse_args()
    import torch
    import rtd3_b200 as rt

    if not torch.cuda.is_available():
        raise SystemExit("rollout_slope.py needs a GPU")
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
    L = rt._lib.lib()
    sp = rt._lib.stream_ptr(dev)
    stream = torch.cuda.current_stream(dev)
    sampler = ClockSampler(0)
    sampler.start()
    Ts = [int(t) for t in args.T.split(",")]
    out = {"card": card, "power_limit_w": power_w, "launches": args.launches, "points": [], "fits": []}
    print("# %s, power limit %s W" % (card, "%.0f" % power_w if power_w else "unknown"))
    for n in [int(v) for v in args.n.split(",")]:
        env = rt.Environment(num_envs=n, seed=1707366464, maps=rt.synthetic_maps(0), device=dev)
        env.reset()
        us = []
        for T in Ts:
            per_buf = T * 2 * n * 4
            R = max(2, int(np.ceil(160e6 / per_buf)) + 1)
            gen = torch.Generator(device=dev).manual_seed(T)
            acts = [torch.rand((T, 2, n), device=dev, generator=gen) * 15 - 7.5 for _ in range(R)]
            trajs = [torch.empty((T, 2, n), device=dev) for _ in range(R)]

            def go(k):
                q = k % R
                rt._lib.check(L.rtd3_env_rollout(env._handle, rt._lib.ptr(env._state[0]), rt._lib.ptr(env._state[1]),
                                                 rt._lib.ptr(acts[q]), rt._lib.ptr(trajs[q]), n, T, sp))

            for k in range(8):
                go(k)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            windows = []
            for r in range(args.reps):
                sampler.in_region = True
                e0.record(stream)
                for k in range(args.launches):
                    go(k)
                e1.record(stream)
                torch.cuda.synchronize(dev)
                sampler.in_region = False
                windows.append(e0.elapsed_time(e1) * 1e3 / args.launches)
            t_us = float(np.median(windows))
            us.append(t_us)
            out["points"].append({"n": n, "T": T, "us_per_launch": round(t_us, 3), "spread_us": round(max(windows) - min(windows), 3)})
            del acts, trajs
        b, a = np.polyfit(np.array(Ts, float), np.array(us), 1)
        clk = sampler.summary()["sm_mhz"]
        fit = {"n": n, "b_ns_per_step": round(b * 1e3, 3), "b_cycles_per_step": round(b * 1e-6 * clk * 1e6, 1) if clk else None,
               "a_us_per_launch": round(a, 2), "sm_mhz": clk,
               "max_residual_us": round(float(np.max(np.abs(np.polyval([b, a], Ts) - us))), 3)}
        out["fits"].append(fit)
        print("n=%-5d  T=%s  us=%s" % (n, Ts, ["%.2f" % u for u in us]))
        print("n=%-5d  b = %.2f ns/step = %s cycles/step at %s MHz, a = %.2f us/launch (max residual %.2f us)" % (
            n, fit["b_ns_per_step"], fit["b_cycles_per_step"], clk, a, fit["max_residual_us"]))
        sys.stdout.flush()
    sampler.stop()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
