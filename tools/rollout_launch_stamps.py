"""Where the fixed cost of a rollout launch goes: %globaltimer stamps of every CTA of the warp-pair kernel at the bench shape.

    python tools/rollout_launch_stamps.py --out DIR [--n 4096] [--T 1000] [--launches 64] [--overlap 0,1] [--json FILE]

Builds librtd3 with -DRTD3_ROLLOUT_STAMPS into DIR (the default build has no stamps), runs `launches` back-to-back
rtd3_env_rollout launches over rotating buffers as bench.py does, and reports per phase the median and max over the CTAs of
the steady launches (the first and last are dropped) of the time since the CTA's start, plus the gap from the last CTA exit of
launch k to the first CTA start of launch k+1 (negative: launch k+1 started before launch k ended) and from that exit to
launch k+1's chain warps starting chunk 0, the critical path between launches.  Phases (rtd3_env.cu, StampPhase): waited = grid_dep_wait returned, table = the chain warp saw the table land, prepped0 = the helper prepped tile 0,
chain0 = the chain warp starts chunk 0, chain_end = it ends the last chunk, last_store = the helper issued the last trajectory
store, exit = the later of the two warps' last stamps.  With one chain/helper pair per CTA (n <= 32 x SMs) every field is one
warp's; with two pairs a field is the later pair's.
"""
import argparse
import glob
import json
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
CSRC = os.path.join(ROOT, "residual-td3-robot-navigation_b200", "csrc")
PHASES = ["start", "waited", "table", "prepped0", "chain0", "chain_end", "last_store", "helper_exit", "chain_exit", "meta"]


def build(out):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    arch = ["-gencode", "arch=compute_100a,code=sm_100a"]
    flags = arch + ["-O3", "-std=c++17", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-DRTD3_ROLLOUT_STAMPS"]
    objdir = os.path.join(out, "stamps_build")
    os.makedirs(objdir, exist_ok=True)
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cu")))
    objs = [os.path.join(objdir, os.path.basename(s)[:-3] + ".o") for s in srcs]
    lib = os.path.join(out, "librtd3_stamps.so")
    deps = srcs + glob.glob(os.path.join(CSRC, "*.cuh")) + [os.path.join(ROOT, "include", "rtd3.h")]
    if os.path.isfile(lib) and os.path.getmtime(lib) > max(os.path.getmtime(d) for d in deps):
        return lib                                         # up to date
    with ThreadPoolExecutor(8) as ex:
        for r in ex.map(lambda so: subprocess.run([nvcc] + flags + ["-c", so[0], "-o", so[1]], capture_output=True, text=True),
                        zip(srcs, objs)):
            if r.returncode:
                raise SystemExit(r.stderr)
    subprocess.run([nvcc] + arch + ["-shared", "-o", lib] + objs, check=True)
    return lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="build directory of the stamped library")
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--T", type=int, default=1000)
    ap.add_argument("--launches", type=int, default=64)
    ap.add_argument("--overlap", default="0,1", help="rtd3_env_set_launch_overlap values to run")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    lib_path = build(args.out)
    import ctypes

    import torch
    import rtd3_b200 as rt
    rt._lib.LIB_PATH = lib_path                            # before the first rt._lib.lib(): the package loads the stamped build
    if not torch.cuda.is_available():
        raise SystemExit("rollout_launch_stamps.py needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    L = rt._lib.lib()
    L.rtd3_rollout_stamps_arm.restype = ctypes.c_int32
    L.rtd3_rollout_stamps_arm.argtypes = [ctypes.c_void_p, ctypes.c_int64]
    words = int(L.rtd3_rollout_stamp_words())
    assert words == len(PHASES)
    card = torch.cuda.get_device_name(dev)
    n, T = args.n, args.T
    env = rt.Environment(num_envs=n, seed=1707366464, maps=rt.synthetic_maps(0), device=dev)
    env.reset()
    per_buf = T * 2 * n * 4
    R = max(2, int(np.ceil(160e6 / per_buf)) + 1)
    gen = torch.Generator(device=dev).manual_seed(0)
    acts = [torch.rand((T, 2, n), device=dev, generator=gen) * 15 - 7.5 for _ in range(R)]
    trajs = [torch.empty((T, 2, n), device=dev) for _ in range(R)]
    sp = rt._lib.stream_ptr(dev)
    out = {"card": card, "n": n, "T": T, "launches": args.launches, "runs": []}
    print("# %s, n=%d T=%d, %d launches" % (card, n, T, args.launches))
    for ov in [int(v) for v in args.overlap.split(",")]:
        L.rtd3_env_set_launch_overlap(ov)

        def go(k):
            q = k % R
            rt._lib.check(L.rtd3_env_rollout(env._handle, rt._lib.ptr(env._state[0]), rt._lib.ptr(env._state[1]),
                                             rt._lib.ptr(acts[q]), rt._lib.ptr(trajs[q]), n, T, sp))

        for k in range(8):
            go(k)
        torch.cuda.synchronize(dev)
        cap = 4 * args.launches * ((n + 31) // 32)
        buf = torch.zeros((cap, words), dtype=torch.int64, device=dev)
        rt._lib.check(L.rtd3_rollout_stamps_arm(ctypes.c_void_p(buf.data_ptr()), cap))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(args.launches):
            go(k)
        e1.record()
        torch.cuda.synchronize(dev)
        rt._lib.check(L.rtd3_rollout_stamps_arm(None, 0))
        us_per_launch = e0.elapsed_time(e1) * 1e3 / args.launches
        rec = buf.cpu().numpy().astype(np.int64)
        rec = rec[rec[:, 0] != 0]
        rec = rec[np.argsort(rec[:, 0], kind="stable")]
        ctas = len(rec) // args.launches
        assert ctas * args.launches == len(rec), (len(rec), args.launches)
        rec = rec.reshape(args.launches, ctas, words)
        exit_ = np.maximum(rec[:, :, PHASES.index("helper_exit")], rec[:, :, PHASES.index("chain_exit")])
        start = rec[:, :, 0]
        steady = slice(1, args.launches - 1)
        row = {"overlap": ov, "us_per_launch": round(us_per_launch, 3), "ctas_per_launch": ctas, "phase_us_since_cta_start": {}}
        for name in PHASES[1:-1] + ["exit"]:
            v = (exit_ if name == "exit" else rec[:, :, PHASES.index(name)])[steady] - start[steady]
            row["phase_us_since_cta_start"][name] = {"median": round(float(np.median(v)) / 1e3, 3), "max": round(float(v.max()) / 1e3, 3)}
        gap = start[1:, :].min(axis=1) - exit_[:-1, :].max(axis=1)
        span = exit_.max(axis=1) - start.min(axis=1)
        spread = start.max(axis=1) - start.min(axis=1)
        row["gap_last_exit_to_next_first_start_us"] = {"median": round(float(np.median(gap)) / 1e3, 3), "min": round(float(gap.min()) / 1e3, 3),
                                                     "max": round(float(gap.max()) / 1e3, 3)}
        # the critical path between launches: from the last CTA exit of launch k to the chain warps of launch k+1 starting chunk 0
        handoff = rec[1:, :, PHASES.index("chain0")] - exit_[:-1, :].max(axis=1, keepdims=True)
        row["last_exit_to_next_chain0_us"] = {"median": round(float(np.median(handoff[steady])) / 1e3, 3),
                                              "max": round(float(handoff[steady].max()) / 1e3, 3)}
        row["launch_span_us"] = {"median": round(float(np.median(span[steady])) / 1e3, 3)}
        row["cta_start_spread_us"] = {"median": round(float(np.median(spread[steady])) / 1e3, 3)}
        out["runs"].append(row)
        print(json.dumps(row))
        sys.stdout.flush()
    L.rtd3_env_set_launch_overlap(1)
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
