"""Policy evaluation (Robot.evaluate) timings: the persistent f16 kernel, the per-step graph path and the Python loop a user would
write without it (get_next_action_testing + step + a float64 distance per step), at T = 1000 test steps.

Grid: n in {4 096, 8 192, 65 536, 262 144}; a 2 x 256 f16 actor and the reference's 3 x 200 fp32 actor; the zero actor (its action
points away from the goal, so every step of every env runs) and an analytic homing actor (residual = -2 base: envs stop early).
Each point is timed in `--windows` windows, the paths alternating inside a window (CUDA events around one whole evaluation, the
environment reset outside); the median is reported, with milliseconds per evaluation and env-steps per second (env-steps = the
steps the envs actually took, the sum of `steps`).  The card's name, power limit and SM clocks are read in the same run.

    python tools/eval_perf.py --out profiles/r7_policy_eval.json

`--episodes E1,E2,...`: the multi-episode form instead.  Per point, one call `evaluate(env, episodes=E)` against the loop it
replaces, E x (env.reset() + evaluate(env)), alternating inside each window and timed with CUDA events around the whole call
or loop (the resets included in both).  Grid: `--sizes` (default 4 096, 16 384, 65 536) x E x zero / homing actor, for the same
two actors.

    python tools/eval_perf.py --episodes 1,16 --out profiles/r8_eval_episodes.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rtd3_b200 as rt  # noqa: E402
from rtd3_b200 import robot as robot_mod  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def set_actor(robot, actor):
    agent = robot.td3_agent
    if actor in ("zero", "homing"):
        agent.flat(0).zero_()
    if actor == "homing":
        net = agent.actor_network
        w1 = net.layer_1.weight
        w1[0, 0], w1[1, 0], w1[2, 1], w1[3, 1] = 1.0, -1.0, 1.0, -1.0
        for k in range(2, agent.layers + 1):
            w = getattr(net, "layer_%d" % k).weight
            for j in range(4):
                w[j, j] = 1.0
        wo = net.output_layer.weight
        wo[0, 0], wo[0, 1], wo[1, 2], wo[1, 3] = -2.0, 2.0, -2.0, 2.0
    agent.sync_transposed()


def python_loop(robot, env, T):
    """What a user writes today: four launches and host work per step, no early stop."""
    goal = env._goal.t()
    best = torch.full((env.num_envs,), float("inf"), dtype=torch.float64, device="cuda")
    success = torch.zeros(env.num_envs, dtype=torch.bool, device="cuda")
    for _ in range(T):
        nxt = env.step(robot.get_next_action_testing(env.robot_state))
        d = torch.linalg.norm(nxt.double() - goal, dim=1)
        best = torch.minimum(best, d)
        success |= d <= 5
    return int(T * env.num_envs)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    work = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), work


SHAPES = {"f16_2x256": (256, 2, "f16"), "fp32_3x200": (200, 3, "fp32")}


def median_point(paths, times, work, **key):
    pt = dict(key, paths={})
    for name in paths:
        med = statistics.median(times[name])
        pt["paths"][name] = {"ms_median": med, "ms_all": times[name], "env_steps": work[name], "env_steps_per_s": work[name] / (med * 1e-3)}
    print(json.dumps(key), {k: round(v["ms_median"], 3) for k, v in pt["paths"].items()}, flush=True)
    return pt


def episodes_main(args, maps, res):
    """One call with E episodes against E x (reset + evaluate), per (actor shape, n, actor, E)."""
    T = args.steps
    res["episodes"] = [int(e) for e in args.episodes.split(",")]
    for shape, (hidden, layers, precision) in SHAPES.items():
        for n in [int(s) for s in args.sizes.split(",")]:
            env = rt.Environment(num_envs=n, seed=5, maps=maps)
            torch.manual_seed(1)
            robot = rt.Robot(env.goal_state, hidden=hidden, layers=layers, seed=3)
            robot.td3_agent.precision = precision
            for actor in ("zero", "homing"):
                set_actor(robot, actor)
                for E in res["episodes"]:
                    def one_call():
                        return robot.evaluate(env, max_steps=T, episodes=E)["steps"]

                    def loop():
                        steps = []
                        for _ in range(E):
                            env.reset()
                            steps.append(robot.evaluate(env, max_steps=T)["steps"])
                        return torch.stack(steps)
                    paths = {"one_call": one_call, "loop": loop}
                    times = {k: [] for k in paths}
                    work = {}
                    for fn in paths.values():                         # warm-up: captures, module loads
                        fn()
                    torch.cuda.synchronize()
                    for _ in range(args.windows):
                        for name, fn in paths.items():
                            torch.cuda.synchronize()
                            ms, w = timed(fn)
                            times[name].append(ms)
                            work[name] = int(w.long().sum())
                    res["points"].append(median_point(paths, times, work, shape=shape, n=n, actor=actor, E=E,
                                                      persistent=bool(robot.td3_agent._f16_ok(n))))
            del robot, env
            torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default=None)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--python-loop-max", type=int, default=1 << 30, help="largest n for which the Python loop is timed")
    ap.add_argument("--episodes", default=None, help="comma-separated E: time evaluate(episodes=E) against the reset + evaluate loop")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs the GPU"
    if args.out is None:
        args.out = os.path.join(ROOT, "profiles", "r8_eval_episodes.json" if args.episodes else "r7_policy_eval.json")
    if args.sizes is None:
        args.sizes = "4096,16384,65536" if args.episodes else "4096,8192,65536,262144"
    T = args.steps
    speed, angle = rt.synthetic_maps(0)
    maps = (speed, (angle * 0.05).astype(np.float32))                # at most 18 degrees of turn: the homing actor reaches goals
    res = {"card": card(), "T": T, "windows": args.windows, "maps": "synthetic_maps(0), angle x 0.05", "points": []}
    if args.episodes:
        episodes_main(args, maps, res)
        return finish(args, res)
    for shape in ("f16_2x256", "fp32_3x200"):
        hidden, layers, precision = (256, 2, "f16") if shape == "f16_2x256" else (200, 3, "fp32")
        for n in [int(s) for s in args.sizes.split(",")]:
            env = rt.Environment(num_envs=n, seed=5, maps=maps)
            torch.manual_seed(1)
            robot = rt.Robot(env.goal_state, hidden=hidden, layers=layers, seed=3)
            robot.td3_agent.precision = precision
            for actor in ("zero", "homing"):
                set_actor(robot, actor)

                def evaluate(persistent, check=True):
                    def f():
                        robot.eval_kernel = persistent
                        robot_mod.EVAL_CHECK_BLOCKS = check
                        r = robot.evaluate(env, max_steps=T)
                        return r["steps"]
                    return f
                paths = {"per_step": evaluate(False), "per_step_no_block_check": evaluate(False, False)}
                if robot.td3_agent._f16_ok(n):
                    paths["persistent"] = evaluate(True)
                if n <= args.python_loop_max:
                    paths["python_loop"] = lambda: python_loop(robot, env, T)
                times = {k: [] for k in paths}
                work = {}
                for name, fn in paths.items():                        # warm-up: captures, module loads
                    env.reset()
                    fn()
                torch.cuda.synchronize()
                for _ in range(args.windows):
                    for name, fn in paths.items():
                        env.reset()
                        torch.cuda.synchronize()
                        ms, w = timed(fn)
                        times[name].append(ms)
                        work[name] = int(w.long().sum()) if isinstance(w, torch.Tensor) else w
                robot_mod.EVAL_CHECK_BLOCKS = True
                pt = {"shape": shape, "n": n, "actor": actor, "paths": {}}
                for name in paths:
                    med = statistics.median(times[name])
                    pt["paths"][name] = {"ms_median": med, "ms_all": times[name], "env_steps": work[name],
                                         "env_steps_per_s": work[name] / (med * 1e-3)}
                res["points"].append(pt)
                print(json.dumps({k: v for k, v in pt.items() if k != "paths"}),
                      {k: round(v["ms_median"], 3) for k, v in pt["paths"].items()}, flush=True)
            del robot, env
            torch.cuda.empty_cache()
    finish(args, res)


def finish(args, res):
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
