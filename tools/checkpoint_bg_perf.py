"""What a background checkpoint costs the run, against the synchronous save, in the configuration of tools/checkpoint_perf.py (a
2 x 256 learner, a filled 1 M-row ring, per-env demonstration sets after three demonstrations; fused ticks, Philox noise, one
host-driven launch sequence per tick, learner off) at N envs (default 8 192 and 65 536), the file in a local temporary directory.

Per N: the synchronous save (the run is stopped until the file is complete); then, alternating, `runs` background saves and `runs`
stretches of the same loop with no save.  For a background save it records the time until the call returns (host clock), the
snapshot's device->device copies (CUDA events around the same staging copies, enqueued on their own after the save), when the
writer starts the file (device->host copies done) and when the file is complete, and the loop's µs per tick while the writer runs:
blocks of `--chunk` ticks, each timed on the host clock up to a synchronise of the current stream only (a device-wide synchronise
would wait for the writer's copies).  The loop with no save runs as many blocks.  `--loop same` times the saved trainer itself;
`--loop throughput` times a second trainer in bench.py's throughput configuration at the same N (shared demonstration set, f16
multi-tick kernel, Philox noise and sampling, learner on at B = 256 x 20 epochs) while the first one's file drains: a loop of tens
of µs per tick, where the writer thread's share of the GIL would show.  Card name, power limit and max SM clock are read in the
same run.
Usage: python tools/checkpoint_bg_perf.py [--envs 8192,65536] [--runs 5] [--loop same|throughput] [--chunk 64]
       [--out profiles/r12_checkpoint_background.json]"""
import argparse
import json
import os
import shutil
import statistics
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
import torch

from checkpoint_perf import build, card, ck, component_bytes, rt


def build_throughput(n):
    """bench.py's throughput loop configuration at n envs, warmed past its first learner update."""
    rs = np.random.RandomState(0)
    tt = np.linspace(0, 1, 3785)[:, None]
    demos = np.concatenate([rs.uniform(5, 95, (1, 2)) * (1 - tt) + rs.uniform(5, 95, (1, 2)) * tt + rs.normal(0, 2.5, (3785, 2)) for _ in range(3)])
    torch.manual_seed(1000)
    env = rt.Environment(num_envs=n, seed=2, maps=rt.synthetic_maps(0))
    robot = rt.Robot(env.goal_state, hidden=256, layers=2, seed=100, buffer_size=max(50000, 8 * n))
    robot.td3_agent.precision = "f16"
    robot.td3_agent.batch_size, robot.td3_agent.num_epochs = 256, 20
    robot.memory.sampler = "philox"
    robot.set_demonstration_states(demos)
    tr = rt.BatchedTrainer(env, robot, noise="philox", graph=True, check_interval=8, fused=True, async_check=True)
    warm = 0
    while warm < 16 or (robot.num_updates < 1 and warm < 400):
        tr.run(8)
        warm += 8
    torch.cuda.synchronize()
    return tr


def loop_block(tr, chunk):
    t = time.perf_counter()
    tr.run(chunk)
    torch.cuda.current_stream().synchronize()
    return (time.perf_counter() - t) / chunk * 1e6


def snapshot_copies_ms(tr):
    live = ck.trainer_state(tr, ck._live)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    staged = ck._map(live, ck._stage)
    e1.record()
    e1.synchronize()
    del staged
    return e0.elapsed_time(e1)


def summary(xs):
    return {"mean": statistics.fmean(xs), "median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}


def measure(n, directory, runs, chunk, loop):
    tr = build(n)
    looped = tr if loop == "same" else build_throughput(n)
    for _ in range(3):
        loop_block(looped, chunk)
    path = os.path.join(directory, "ckpt_%d.pt" % n)
    sizes = component_bytes(tr.state_dict())
    res = {"num_envs": n, "bytes": sizes["total"], "loop": loop, "chunk_ticks": chunk}
    torch.cuda.synchronize()
    t = time.perf_counter()
    rt.save_checkpoint(path, tr)
    res["sync_save_s"] = time.perf_counter() - t
    os.unlink(path)

    stamps = {}
    real = ck._atomic_save

    def stamped(payload, file):
        stamps["write_start"] = time.perf_counter()
        real(payload, file)
        stamps["write_end"] = time.perf_counter()
    ck._atomic_save = stamped
    bg, plain = [], []
    try:
        for r in range(runs):
            torch.cuda.synchronize()
            stamps.clear()
            t0 = time.perf_counter()
            p = rt.save_checkpoint(path, tr, background=True)
            t_return = time.perf_counter() - t0
            during = []
            while not p.done():
                during.append(loop_block(looped, chunk))
            p.wait()
            t_done = stamps["write_end"] - t0
            os.unlink(path)
            copies = snapshot_copies_ms(tr)
            bg.append({"call_returns_s": t_return, "snapshot_copies_ms": copies, "device_to_host_done_s": stamps["write_start"] - t0,
                       "file_complete_s": t_done, "blocks_during_drain": len(during),
                       "us_per_tick_during_drain": statistics.fmean(during) if during else None})
            base = [loop_block(looped, chunk) for _ in range(max(len(during), 1))]
            plain.append({"blocks": len(base), "us_per_tick": statistics.fmean(base)})
            print(json.dumps({"num_envs": n, "loop": loop, "run": r, "background": bg[-1], "no_save": plain[-1]}), flush=True)
    finally:
        ck._atomic_save = real
    res["background_runs"], res["no_save_runs"] = bg, plain
    stopped = [b["call_returns_s"] + b["snapshot_copies_ms"] * 1e-3 for b in bg]
    res["summary"] = {"sync_save_s": res["sync_save_s"],
                      "call_returns_s": summary([b["call_returns_s"] for b in bg]),
                      "snapshot_copies_ms": summary([b["snapshot_copies_ms"] for b in bg]),
                      "run_stopped_s (call + snapshot copies)": summary(stopped),
                      "file_complete_s": summary([b["file_complete_s"] for b in bg]),
                      "us_per_tick_during_drain": summary([b["us_per_tick_during_drain"] for b in bg if b["us_per_tick_during_drain"]]),
                      "us_per_tick_no_save": summary([p["us_per_tick"] for p in plain]),
                      "sync_over_background_stop": res["sync_save_s"] / statistics.median(stopped)}
    del tr, looped
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="8192,65536")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--loop", choices=("same", "throughput"), default="same")
    ap.add_argument("--chunk", type=int, default=64)
    ap.add_argument("--dir", default=None)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("checkpoint_bg_perf needs the GPU")
    directory = a.dir or tempfile.mkdtemp(prefix="rtd3_ckpt_bg_perf_")
    out = {"card": card(), "results": []}
    try:
        for n in (int(x) for x in a.envs.split(",")):
            r = measure(n, directory, a.runs, a.chunk, a.loop)
            out["results"].append(r)
            print(json.dumps({"num_envs": n, "summary": r["summary"]}), flush=True)
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
