"""Checkpoint size and save / load times of a BatchedTrainer at user scale: N envs (default 8 192 and 65 536), a 2 x 256 learner, a
1 M-row replay ring (filled) and per-env demonstration sets after the reference's three demonstrations (11 355 float64 states per env).

Reports, per N: checkpoint bytes by component; save = device->host (`state_dict`, which synchronises) + file write (atomic
`torch.save`); load = file read (`torch.load`) + host->device and rebuilds (`load_state_dict`), with the rebuilds (per-env grids,
map tables, derived weight copies) also timed on their own; and the card's name and power limit, read in the same run.
Usage: python tools/checkpoint_perf.py [--envs 8192,65536] [--dir DIR] [--out checkpoint_perf.json]"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import rtd3_b200 as rt
from importlib import import_module
from oracle import env_oracle as eo

ck = import_module("residual-td3-robot-navigation_b200.checkpoint")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def build(n):
    env = rt.Environment(num_envs=n, seed=1, maps=eo.synthetic_maps(0))
    robot = rt.Robot(env._goal.t(), hidden=256, layers=2, seed=1, buffer_size=1 << 20)
    robot.episodes_per_update = 1 << 30
    robot.memory.sampler = "philox"                     # the exact sampler draws from at most 56 000 rows
    tr = rt.BatchedTrainer(env, robot, fused=True, noise="philox")
    g = torch.Generator(device="cuda").manual_seed(0)
    for _ in range(3):                                  # three demonstrations per env: the sets reach their final size
        walk = torch.cumsum(torch.rand((n, 200, 2), device="cuda", generator=g) - 0.5, 1) + env._state.t()[:, None]
        robot.process_demonstration(walk.clamp(0, 99).contiguous(), torch.zeros_like(walk), None)
    tr.run(4)
    rows = 1 << 20                                      # the ring full
    s = torch.rand((rows, 2), device="cuda", generator=g) * 99
    rb = robot.memory
    rb.push(s, s * 0.01, -s[:, 0], s, torch.zeros(rows, dtype=torch.bool, device="cuda"))
    robot.td3_agent.td3_update(rb)
    torch.cuda.synchronize()
    return tr


def component_bytes(sd):
    out = {}

    def add(name, v):
        if isinstance(v, torch.Tensor):
            out[name] = out.get(name, 0) + v.numel() * v.element_size()
        elif isinstance(v, dict):
            for x in v.values():
                add(name, x)
        elif isinstance(v, (list, tuple)):
            for x in v:
                add(name, x)
    add("trainer", {k: sd[k] for k in ("tensors", "host")})
    add("environment", sd["env"])
    r = sd["robot"]
    sets = {k: v for k, v in r["tensors"].items() if k.startswith("_env_demo")}
    add("robot per-env demonstration sets", sets)
    add("robot episode state and RNG", {k: v for k, v in r["tensors"].items() if k not in sets})
    add("robot host (shared set, counters)", r["host"])
    add("replay ring", r["memory"])
    add("learner (arena, Adam)", r["td3_agent"])
    out["total"] = sum(out.values())
    return out


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t


def measure(n, directory):
    tr = build(n)
    sd, t_d2h = timed(tr.state_dict)
    sizes = component_bytes(sd)
    res = {"num_envs": n, "bytes": sizes}
    free = shutil.disk_usage(directory).free
    path = os.path.join(directory, "ckpt_%d.pt" % n)
    if free > 2 * sizes["total"]:
        _, t_write = timed(lambda: ck._atomic_save({"meta": ck._summary(tr), "state": sd}, path))
        res["file_bytes"] = os.path.getsize(path)
        payload, t_read = timed(lambda: torch.load(path, map_location="cpu", weights_only=True))
        os.unlink(path)
        sd = payload["state"]
    else:
        t_write = t_read = None
        res["file"] = "not measured: %.1f GB free in %s" % (free / 1e9, directory)
    _, t_load = timed(lambda: tr.load_state_dict(sd))
    d = tr.robot._env_demo

    def rebuilds():
        rt._lib.check(rt._lib.lib().rtd3_robot_demo_grids(rt._lib.ptr(d["sets"]), rt._lib.ptr(d["count"]), d["cap"], n, rt._lib.ptr(d["sorted"]),
                                                          rt._lib.ptr(d["cells"]), rt._lib.stream_ptr()), "robot_demo_grids")
        tr.env._install_maps(torch.from_numpy(tr.env.dynamics_speed), torch.from_numpy(tr.env.dynamics_angle), None)
        ck._rebuild_weights(tr.robot.td3_agent)
    _, t_rebuild = timed(rebuilds)
    _, t_grids = timed(lambda: rt._lib.check(rt._lib.lib().rtd3_robot_demo_grids(
        rt._lib.ptr(d["sets"]), rt._lib.ptr(d["count"]), d["cap"], n, rt._lib.ptr(d["sorted"]), rt._lib.ptr(d["cells"]), rt._lib.stream_ptr()), "grids"))
    res["seconds"] = {"save_device_to_host": t_d2h, "save_file_write": t_write, "load_file_read": t_read,
                      "load_host_to_device_and_rebuilds": t_load, "rebuilds_alone": t_rebuild, "demo_grids_kernel_alone": t_grids}
    del tr, sd
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="8192,65536")
    ap.add_argument("--dir", default=None)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("checkpoint_perf needs the GPU")
    directory = a.dir or tempfile.mkdtemp(prefix="rtd3_ckpt_perf_")
    out = {"card": card(), "results": []}
    try:
        for n in (int(x) for x in a.envs.split(",")):
            r = measure(n, directory)
            out["results"].append(r)
            print(json.dumps(r), flush=True)
    finally:
        if a.dir is None:
            shutil.rmtree(directory, ignore_errors=True)
    out["card"]["after"] = card()["nvidia_smi"]
    print(json.dumps(out["card"]))
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
