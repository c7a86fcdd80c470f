#!/usr/bin/env python
"""bench.py - headline measurement of the hot path (BASELINE.json: env-steps/sec; TD3 updates/sec rides along).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

Workload at every N (weak scaling, per GPU): BASELINE.json configs[1] - a batched dynamics rollout of 4096 envs,
random actions U(-7.5, 7.5), 1000 steps.  One bench "step" = LAUNCHES_PER_STEP such rollouts back to back (one launch of the
rollout kernel each), so that the timed window is tens of milliseconds and not a single millisecond of launch jitter.
Inputs rotate through enough distinct action/trajectory buffers that the footprint exceeds the 126 MB L2.
Both arms run the SAME workload: start states and actions come from numpy generators seeded per rank (make_workload), so the
CPU arm steps exactly the envs, from exactly the states, with exactly the actions the GPU arm does.
Prints ONE JSON line on rank 0 (see the task contract); `--impl reference` times the CPU oracle port instead.
"""
import argparse
import json
import multiprocessing as mp
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS = 4096          # configs[1]
T_STEPS = 1000       # configs[1]
LAUNCHES_PER_STEP = 64   # rollouts per bench step: 64 x ~47 us = 3 ms per step, 60 ms for a 20-step run
E2E_CALLS_PER_STEP = 8   # host-buffer calls per e2e step: 8 x ~0.9 ms
ACTION_RANGE = 7.5   # SURVEY.md 8(d) config 2
SEED = 1707366464
ROLL_BYTES_PER_ENV_STEP = 16   # 8 B action read + 8 B state written; state stays in registers (DESIGN.md)
STEP_BYTES_PER_ENV_STEP = 24   # single-step kernel: state in 8 + action in 8 + state out 8
WORKLOAD = "batched dynamics rollout: %d envs x %d steps per GPU, random actions U(-7.5,7.5) (configs[1])" % (ENVS, T_STEPS)


def make_workload(rank, n, T, buffers):
    """Start states `[n,2]` and `buffers` action sets `[T,2,n]` (float32) of rank `rank`, identical in both arms."""
    rs = np.random.RandomState((SEED + rank) % (2 ** 32))
    starts = rs.uniform(0, 98.9999, (n, 2)).astype(np.float32)
    acts = [rs.uniform(-ACTION_RANGE, ACTION_RANGE, (T, 2, n)).astype(np.float32) for _ in range(buffers)]
    return starts, acts


DUMP_BYTES = 60 * 10 ** 6   # --dump-outputs stays under 64 MB, .npy headers included


def dump_outputs(out_dir, state, traj):
    """What a caller of rtd3_env_rollout receives from the last launch of the last timed step: the final state `[2,n]` and the
    trajectory `[T,2,n]` (float32).  A trajectory over the budget keeps a fixed, seeded sample of env columns."""
    T, _, n = traj.shape
    keep = min(n, (DUMP_BYTES - state.numel() * 4) // (T * 2 * 4))
    traj = traj.cpu().numpy()
    if keep < n:
        traj = traj[:, :, np.sort(np.random.RandomState(0).choice(n, keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "final_state.npy"), state.cpu().numpy())
    np.save(os.path.join(out_dir, "trajectory.npy"), np.ascontiguousarray(traj))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1590.0)), "measured"
    return 6650.0, 1590.0, "fallback"


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.in_region = False
        self._stop = threading.Event()
        self.ok = False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._stop.is_set():
            try:
                mhz = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                try:
                    r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                if self.in_region:
                    self.samples.append(mhz)
                    for bit, name in self.REASONS.items():
                        if r & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def stop(self):
        self._stop.set()

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs NVML reports as local to GPU `index`: pinned host buffers are then first-touched on the GPU's
    own NUMA node, so the PCIe DMA of the host-buffer path does not cross the socket interconnect.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return 0


# ------------------------------------------------------------------------------------------ CPU arm
_CPU_WORK = {}


def _cpu_worker(args):
    """Scalar oracle port: the reference's own per-env Python loop (environment.py:122-127) on this worker's envs, from the
    workload's start states with the workload's actions (inherited from the parent through fork)."""
    lo, hi, t0s, t1s = args
    from oracle import env_oracle as eo
    speed, angle = _CPU_WORK["maps"]
    states, actions = _CPU_WORK["starts"], _CPU_WORK["actions"]
    t0 = time.perf_counter()
    for i in range(lo, hi):
        s = states[i].astype(np.float64)
        for t in range(t0s, t1s):
            s = eo.step_scalar(speed, angle, s, actions[t, :, i])
    return time.perf_counter() - t0, (hi - lo) * (t1s - t0s)


def cpu_env_steps(envs, t_begin, t_end, procs, pool=None):
    """env-steps/s of the oracle port over `procs` worker processes (each one GIL-bound core): envs 0..envs-1, rollout steps
    t_begin..t_end-1 of the workload."""
    bounds = np.linspace(0, envs, procs + 1).astype(int)
    jobs = [(int(bounds[k]), int(bounds[k + 1]), t_begin, t_end) for k in range(procs) if bounds[k + 1] > bounds[k]]
    t0 = time.perf_counter()
    if pool is None:
        res = [_cpu_worker(j) for j in jobs]
    else:
        res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    total = sum(r[1] for r in res)
    return total / wall, wall, total


def _cpu_prepare():
    from oracle import env_oracle as eo
    starts, acts = make_workload(0, ENVS, T_STEPS, 1)
    _CPU_WORK.update(maps=eo.synthetic_maps(0), starts=starts, actions=acts[0])


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    procs = os.cpu_count() or 1
    # 4096 envs x 48 of the 1000 rollout steps per bench step, walking through the workload's steps: a bounded sample (~0.12 s on
    # 16 cores) long enough that the workers' per-job set-up does not count against the reference
    t_sample = 48
    _cpu_prepare()
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        for k in range(args.warmup):
            cpu_env_steps(ENVS, 0, t_sample, procs, pool)
        t0 = time.perf_counter()
        total = 0
        for k in range(args.steps):
            lo = (k * t_sample) % (T_STEPS - t_sample)
            _, _, n = cpu_env_steps(ENVS, lo, lo + t_sample, procs, pool)
            total += n
        wall = time.perf_counter() - t0
    value = total / wall
    sample = "%d envs x %d of the %d rollout steps per bench step (the GPU arm's start states and actions), scalar oracle port (oracle/env_oracle.py step_scalar), %d processes" % (
        ENVS, t_sample, T_STEPS, procs)
    line = {
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": procs, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------ TD3 legs
TD3_SHAPES = [  # (label, batch, hidden, layers, epochs): configs[2] benchmark shape, the reference's own shape, configs[4] large batch
    ("B256_2x256", 256, 256, 2, 100),
    ("B100_3x200_reference_shape", 100, 200, 3, 100),
    ("B8192_2x256", 8192, 256, 2, 20),
    ("B8192_2x256_tf32_tcgen05", 8192, 256, 2, 20),      # same shape on the tensor-core learner (opt-in precision="tf32")
    ("B65536_2x256_tf32_tcgen05", 65536, 256, 2, 10),
]
FP32_FFMA_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # nominal: 148 SMs x 128 lanes x 2 flop x 1.965 GHz


def td3_flops_per_epoch(B, H, L):
    """Algorithmic FLOPs (2*MAC) of one epoch = critic step + 1/2 actor step (SURVEY.md 8a-7/8: fwd + bwd incl. targets)."""
    actor = 2 * H + (L - 1) * H * H + H * 2
    critic = 4 * H + (L - 1) * H * H + H * 1
    critic_step = actor + 2 * critic + 2 * 3 * critic          # target actor, 2 target critics, 2 x (fwd + bwd(dX + dW))
    actor_step = 3 * actor + critic + critic                   # actor fwd + bwd(dX+dW), critic-1 fwd, critic-1 bwd (dX only)
    return 2.0 * B * (critic_step + 0.5 * actor_step)


def cpu_td3_epochs_per_sec(B, H, L, epochs):
    """The oracle port (numpy float32, BLAS threads as configured) of TD3.td3_update on a synthetic replay."""
    from oracle import td3_oracle as to
    rs = np.random.RandomState(0)
    w = [to.kaiming_uniform_params(rs, 2, H, L, 2), to.kaiming_uniform_params(rs, 4, H, L, 1), to.kaiming_uniform_params(rs, 4, H, L, 1)]
    orc = to.TD3Oracle(w[0], w[1], w[2], hidden=H, layers=L)
    n = 10000
    rb = to.ReplayOracle(n)
    rb.s[:] = rs.uniform(0, 98.9999, (n, 2)); rb.a[:] = rs.uniform(-5, 5, (n, 2)); rb.s2[:] = np.clip(rb.s + rb.a, 0, 98.9999)
    rb.r[:] = -np.linalg.norm(rb.s2 - np.array([80, 20], np.float32), axis=1); rb.size = n
    # index draws through numpy's own C implementation of the legacy shuffle, as the reference does (robot.py:111)
    t0 = time.perf_counter()
    for e in range(epochs):
        idx = rs.choice(n, B, replace=False) if B <= n else rs.randint(0, n, B)
        orc.train_critic(*rb.gather(idx), rs.normal(size=(B, 2)).astype(np.float32))
        if e % 2 == 0:
            idx = rs.choice(n, B, replace=False) if B <= n else rs.randint(0, n, B)
            orc.train_actor(rb.gather(idx)[0])
            orc.polyak_all()
    return epochs / (time.perf_counter() - t0)


def dp_step_form(agent, B, tf32, world):
    """Which form the optimiser step of the data-parallel learner takes (decided inside rtd3_td3_update, csrc/rtd3_td3.cu)."""
    if world == 1:
        return None
    if getattr(agent, "dp_collective", None) != "p2p":
        return "rtd3_allreduce_grads (NCCL, in the update graph) + optimiser kernel"
    if not tf32 and B <= 512 and int(os.environ.get("RTD3_P2P_FUSE", "2")) >= 2:
        return ("weight-gradient kernels exchange their own gradient tiles over peer memory ({value, step} lines, no fence, no all-reduce launch; %s) "
                "and apply Adam / Polyak to the sums" % ("all to all" if world <= 2 else "reduce-scatter + all-gather by block owner"))
    return "p2p_allreduce_adam_kernel: peer-memory all-reduce that applies Adam / Polyak to the sums (one cooperative launch per optimiser step)"


def bench_td3(rt, torch, dev, world, rank, cpu):
    import torch.distributed as dist
    out = []
    pg = dist.group.WORLD if world > 1 else None
    for label, B, H, L, epochs in TD3_SHAPES:
        torch.manual_seed(rank)                           # ranks start from different weights: the constructor broadcasts rank 0's
        agent = rt.TD3(rt.Residual_Actor_Network(H, L), rt.Residual_Critic_Network(H, L), rt.Residual_Critic_Network(H, L),
                       batch_size=B, num_epochs=epochs, device=dev, process_group=pg)
        tf32 = label.endswith("tcgen05")
        if tf32:
            agent.precision = "tf32"
        n = 10000 if B <= 10000 else 2 * B                # the reference's buffer size (robot.py:36) unless the batch needs more rows
        rb = rt.ReplayBuffer(n, device=dev, seed=rank)
        g = torch.Generator(device=dev).manual_seed(rank)
        s = torch.rand((n, 2), device=dev, generator=g) * 98.9999
        a = torch.rand((n, 2), device=dev, generator=g) * 10 - 5
        s2 = (s + a).clamp(0, 98.9999)
        r = -torch.linalg.norm(s2 - torch.tensor([80., 20.], device=dev), dim=1)
        rb.push(s, a, r, s2, (torch.arange(n, device=dev) % 50) == 49)
        if B > 10000:
            rb.sampler = "philox"                         # throughput sampler (the exact MT19937 protocol is timed on the shapes above)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        reps, ms_s, ms_u, ms_full = 4, [], [], []
        for rep in range(reps):                           # rep 0 captures the graphs / warms up
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
            ev[0].record()
            idx = rb.sample_indices(B, epochs + (epochs + 1) // 2)      # the index draw alone ...
            ev[1].record()
            agent.td3_update(rb, idx=idx)                               # ... the update alone ...
            ev[2].record()
            torch.cuda.synchronize(dev)
            ev[3].record()
            agent.td3_update(rb)                                        # ... and the call a user makes: draw + update, pipelined
            ev[4].record()
            torch.cuda.synchronize(dev)
            if rep > 0:
                ms_s.append(ev[0].elapsed_time(ev[1])); ms_u.append(ev[1].elapsed_time(ev[2])); ms_full.append(ev[3].elapsed_time(ev[4]))
        t = torch.tensor([float(np.median(ms_s)), float(np.median(ms_u)), float(np.median(ms_full))], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_sample, ms_update, ms_call = float(t[0]), float(t[1]), float(t[2])
        flops = td3_flops_per_epoch(B * world, H, L) * epochs
        row = {"shape": label, "global_batch": B * world, "epochs": epochs, "sampler": rb.sampler,
               "update_kernel": ("tcgen05 step kernels" if tf32 else ("persistent cooperative kernel (rtd3_td3_update_coop)" if agent._coop_ok(B)
                                                                     else ("cluster step kernels (rtd3_td3_update: 4-CTA clusters, columns split, st.async hand-over)"
                                                                           if rt._lib.lib().rtd3_td3_cluster_supported(agent._handle, B)
                                                                           else "row-tile step kernels (rtd3_td3_update)"))),
               "dp_collective": getattr(agent, "dp_collective", None) if world > 1 else None,
               "dp_step": dp_step_form(agent, B, tf32, world),
               "update_ms": round(ms_update, 3), "sampler_ms": round(ms_sample, 3), "us_per_epoch": round(1e3 * ms_update / epochs, 2),
               "td3_update_call_ms": round(ms_call, 3), "updates_per_sec": epochs / (ms_call * 1e-3),
               "updates_per_sec_update_only": epochs / (ms_update * 1e-3),
               "precision": "tf32 (tcgen05.mma kind::tf32, fp32 accumulate in TMEM)" if tf32 else "fp32 (FFMA)"}
        tfl = flops / (ms_update * 1e-3) / 1e12
        if tf32:
            row["tflops_tf32"] = tfl
            row["frac_of_tf32_peak"] = tfl / (load_peaks()[1] / 2 * world)      # TF32 dense = half the measured bf16 figure
        else:
            row["tflops_fp32"] = tfl
            row["frac_of_nominal_fp32_peak"] = tfl / (FP32_FFMA_PEAK_TFLOPS * world)
        # roofline-shaped object of this leg: algorithmic flops of an epoch (td3_flops_per_epoch) over the measured epoch time, against
        # the peak of the pipe the kernels use (TF32: half the measured dense bf16 figure; fp32 FFMA: nominal, no measured figure exists)
        peak = (load_peaks()[1] / 2 if tf32 else FP32_FFMA_PEAK_TFLOPS) * world
        row["roofline"] = {"bound": "tensor" if tf32 else "fp32_ffma", "achieved": tfl, "peak": peak, "unit": "TFLOP/s", "frac": tfl / peak,
                           "flops_per_epoch": flops / epochs, "us_per_epoch": 1e3 * ms_update / epochs,
                           "peak_kind": "measured bf16 / 2" if tf32 else "nominal 148 SM x 128 lanes x 2 x 1.965 GHz"}
        if cpu and rank == 0 and world == 1 and not tf32:
            e_cpu = 40 if B <= 256 else 4
            row["cpu_port_updates_per_sec"] = cpu_td3_epochs_per_sec(B, H, L, e_cpu)
        if world > 1:
            from rtd3_b200.trainer import replicas_identical
            row["replicas_identical"] = replicas_identical(agent, pg)
        out.append(row)
        del agent, rb
    return out


def bench_forward(rt, torch, dev):
    """Actor forward (2 -> 256 -> 256 -> 2) of the act hook at rollout-sized batches: fp32 FFMA kernel vs the tcgen05 / TMEM
    TF32 kernel (weights streamed per tile) and the f16 kernel (weights resident; both opt-in throughput modes).  Tensor-pipe
    roofline: the measured dense bf16 peak for 16-bit operands, half of it as the TF32 reference."""
    H, L = 256, 2
    agent = rt.TD3(rt.Residual_Actor_Network(H, L), rt.Residual_Critic_Network(H, L), rt.Residual_Critic_Network(H, L), device=dev)
    agent.sync_transposed()
    _, bf16_peak, _ = load_peaks()
    rows = []
    for B in (65536, 1 << 20):
        xs = [torch.rand((B, 2), device=dev) * 100 - 50 for _ in range(3)]
        flops = 2.0 * B * (2 * H + (L - 1) * H * H + 2 * H)
        for precision in ("fp32", "tf32", "f16"):
            agent.precision = precision
            for k in range(3):
                agent.forward(0, xs[k])
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 10
            e0.record()
            for k in range(reps):
                agent.forward(0, xs[k % 3])
            e1.record()
            torch.cuda.synchronize(dev)
            us = e0.elapsed_time(e1) * 1e3 / reps
            row = {"batch": B, "precision": precision, "us": round(us, 1), "rows_per_sec": B / (us * 1e-6), "tflops": flops / us / 1e6}
            if precision == "tf32":
                row["frac_of_tf32_peak"] = row["tflops"] / (bf16_peak / 2)
            elif precision == "f16":
                row["frac_of_16bit_dense_peak"] = row["tflops"] / bf16_peak
                row["kernel"] = "mlp_forward_f16_kernel: fp16 operands, hidden weight resident in shared memory, tcgen05.mma.kind::f16"
            else:
                row["frac_of_nominal_fp32_peak"] = row["tflops"] / FP32_FFMA_PEAK_TFLOPS
            rows.append(row)
    return rows


def bench_single_env(rt, torch, dev):
    """configs[0]: the reference's own run - robot-learning.py's update(dt) for ONE env, seeded, default demo budget - through the
    drop-in classes (`trainer.DriverLoop`: Environment / Robot hooks one call per tick, host <-> device copies and a sync per hook).
    Wall clock per tick by kind, beside the survey-time figures of the unmodified reference on CPU (BASELINE.md section 2; not re-timed
    here: the reference cannot travel to the GPU box)."""
    import numpy as _np
    from rtd3_b200.trainer import DriverLoop
    speed, angle = rt.synthetic_maps(0)
    torch.manual_seed(0)
    t_build = time.perf_counter()
    loop = DriverLoop.from_seed(1707366464, maps=(speed, angle))
    build_s = time.perf_counter() - t_build
    robot = loop.robot
    upd = {"n": 0, "s": 0.0, "each": []}
    real_update = robot.td3_agent.td3_update

    def timed_update(*a, **kw):
        t0 = time.perf_counter()
        out = real_update(*a, **kw)
        torch.cuda.synchronize(dev)
        upd["n"] += 1
        upd["s"] += time.perf_counter() - t0
        upd["each"].append(time.perf_counter() - t0)
        return out
    robot.td3_agent.td3_update = timed_update
    per_kind = {}
    t_run = time.perf_counter()
    ticks = 0
    while not loop.finished and ticks < 5000:
        u0 = upd["s"]
        t0 = time.perf_counter()
        kind = loop.update()
        dt = time.perf_counter() - t0 - (upd["s"] - u0)              # the learner update of an episode end is reported separately
        per_kind.setdefault(kind or "none", []).append(dt)
        ticks += 1
    total_s = time.perf_counter() - t_run
    row = {"config": "configs[0]: reference robot-learning.py loop, single env, seed 1707366464, default demo budget, synthetic maps",
           "ticks": ticks, "total_s": round(total_s, 3), "build_s": round(build_s, 3), "success": bool(loop.success), "td3_updates": upd["n"],
           "ms_per_td3_update_100_epochs": {"median": round(1e3 * float(_np.median(upd["each"])), 3) if upd["each"] else None,
                                            "first_call_with_graph_capture": round(1e3 * upd["each"][0], 3) if upd["each"] else None},
           "ms_per_tick_by_kind": {k: {"n": len(v), "median_ms": round(1e3 * float(_np.median(v)), 4), "mean_ms": round(1e3 * float(_np.mean(v)), 4)}
                                   for k, v in per_kind.items()},
           "reference_cpu_survey": {"training_tick_ms": 4.4, "td3_update_100_epochs_ms": "720-1270", "get_demonstration_s": 3.5,
                                    "source": "BASELINE.md section 2 (unmodified reference, survey container, 8 vCPU); not re-timed on this box"}}
    return row


def bench_full_loop(rt, torch, dev, world, rank):
    """configs[3]: the act -> step -> transition -> (episodes ended: TD3 update) loop, gradients all-reduced across ranks.
    8192 envs per GPU (65536 over 8 GPUs) and, for the per-GPU ceiling, 65536 envs per GPU.  Every row states its mode:
      throughput - Philox exploration noise in the tick kernel, f16 tensor-core actor forward, Philox replay sampling (with replacement);
      exact      - the parity path: per-env numpy-legacy MT19937 noise, fp32 forward, exact np.random.choice index draws;
      reference cadence - exact mode with the reference's own update (100 epochs x B 100, 3 x 200 networks, robot.py:46-54)."""
    import torch.distributed as dist
    from rtd3_b200.trainer import replicas_identical
    pg = dist.group.WORLD if world > 1 else None
    rows = []
    rs = np.random.RandomState(0)
    tt = np.linspace(0, 1, 3785)[:, None]                # 3 x 3785 = the 11 355 demonstration states the reference holds after its 3 demos
    demos = np.concatenate([rs.uniform(5, 95, (1, 2)) * (1 - tt) + rs.uniform(5, 95, (1, 2)) * tt + rs.normal(0, 2.5, (3785, 2)) for _ in range(3)])
    configs = [  # (envs per GPU, mode, hidden, layers, batch, epochs per update)
        (8192, "throughput", 256, 2, 256, 20),
        (8192, "exact", 256, 2, 256, 20),
        (8192, "reference cadence", 200, 3, 100, 100),
        (65536, "throughput", 256, 2, 256, 20),
    ]
    for n, mode, H, Lh, B, E in configs:
        torch.manual_seed(1000 + rank)
        env = rt.Environment(num_envs=n, seed=SEED + rank * n, device=dev, maps=rt.synthetic_maps(0))
        thr = mode == "throughput"
        # throughput: a ring that holds eight ticks of every env (the multi-tick kernel's bound); exact: the reference's BUFFER_SIZE
        # (robot.py:36) - the exact index draw shuffles the whole ring per minibatch, as np.random.choice does
        robot = rt.Robot(env.goal_state, hidden=H, layers=Lh, seed=100 + rank, device=dev, process_group=pg,
                         buffer_size=max(50000, 8 * n) if thr else 10000)
        robot.td3_agent.precision = "f16" if thr else "fp32"
        robot.td3_agent.batch_size = B
        robot.td3_agent.num_epochs = E
        robot.memory.sampler = "philox" if thr else "mt19937"
        robot.set_demonstration_states(demos)
        tr = rt.BatchedTrainer(env, robot, noise="philox" if thr else "mt19937", graph=True, check_interval=8, fused=True, async_check=True)
        warm = 0
        while warm < 16 or (robot.num_updates < 1 and warm < 400):      # past the first learner update: its one-time graph
            tr.run(8)                                                  # capture (tens of ms) is not part of the steady state
            warm += 8
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ticks, upd0, steps0 = 480, robot.num_updates, int(tr.steps_bought.sum())   # long enough to average over the update cadence
        e0.record()
        tr.run(ticks)
        e1.record()
        torch.cuda.synchronize(dev)
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        st = torch.tensor([float(int(tr.steps_bought.sum()) - steps0)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(st)
        ms = float(t[0])
        updates = robot.num_updates - upd0
        agent = robot.td3_agent
        row = {"envs_per_gpu": n, "envs_total": n * world, "mode": mode, "networks": "%d x %d" % (Lh, H), "actor_forward": agent.precision,
               "exploration_noise": tr.noise, "replay_sampler": robot.memory.sampler, "tick": "fused", "ticks": ticks, "ms_per_tick": ms / ticks,
               "env_steps_per_sec": float(st[0]) / (ms * 1e-3), "td3_updates_in_window": updates, "td3_epochs_per_update": E,
               "td3_batch_per_gpu": B, "td3_epochs_per_sec": updates * E / (ms * 1e-3),
               # sampled minibatch rows per env-step collected (the reference: 100 epochs x 1.5 x 100 rows per ~60-step episode = ~250)
               "update_to_data_ratio": updates * E * 1.5 * B * world / max(float(st[0]), 1.0),
               "episodes_per_update": robot.episodes_per_update * world, "update_check": "asynchronous (counter snapshot of the previous block)",
               "replay_rows_per_gpu": len(robot.memory), "demo_states": int(demos.shape[0]),
               "update_kernel": "persistent cooperative kernel" if agent._coop_ok(B) else "per-step kernels",
               "dp_collective": getattr(agent, "dp_collective", None) if world > 1 else None,
               "tick_form": ("eight ticks per launch of the multi-tick kernel rtd3_tick_run_f16 (actor forward inside)" if tr._multi_tick_ok() else
                             "three launches per tick (rtd3_tick_pre / actor forward / rtd3_tick_post), eight ticks per CUDA graph")}
        if world > 1:
            row["replicas_identical"] = replicas_identical(agent, pg)
        rows.append(row)
        del tr, robot, env
        import gc
        gc.collect()                                     # finalise the handles (cudaFree) now, not inside the next config's graph capture
    return rows

# ------------------------------------------------------------------------------------------ GPU arm
def run_b200(args):
    # ---- CPU baseline (rank 0, N=1 only): scalar oracle port on all host cores, bounded sample of the SAME workload
    cpu = None
    if int(os.environ.get("RANK", "0")) == 0 and int(os.environ.get("WORLD_SIZE", "1")) == 1 and not args.no_cpu:
        procs = os.cpu_count() or 1
        _cpu_prepare()
        ctx = mp.get_context("fork")
        with ctx.Pool(procs) as pool:
            cpu_env_steps(procs * 4, 0, 8, procs, pool)                                # warm the workers
            t_sample = 200                                                             # ~13 core-seconds of the reference loop
            v_all, wall, total = cpu_env_steps(ENVS, 0, t_sample, procs, pool)
        v_one, _, _ = cpu_env_steps(64, 0, 16, 1, None)
        # the same arithmetic vectorised over the envs in numpy (not how the reference runs, reported for context)
        from oracle import env_oracle as eo
        sp_, an_ = _CPU_WORK["maps"]
        st_ = _CPU_WORK["starts"].astype(np.float64)
        t0_ = time.perf_counter()
        for t_ in range(50):
            st_ = eo.step_batch(sp_, an_, st_, _CPU_WORK["actions"][t_].T)
        v_vec = ENVS * 50 / (time.perf_counter() - t0_)
        cpu = {"value": v_all, "unit": "env-steps/s", "cores": procs, "kind": "port",
               "sample": "%d envs x the first %d of the %d rollout steps (%.1f s wall), the GPU arm's start states and actions, scalar oracle port in %d processes; 1 process: %.3g env-steps/s"
                         % (ENVS, t_sample, T_STEPS, wall, procs, v_one),
               "vectorised_numpy_1core": v_vec}

    import torch
    import torch.distributed as dist
    import rtd3_b200 as rt

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    hbm_peak, _, peak_kind = load_peaks()

    bind_to_gpu_numa_node(local_rank)                    # pinned host buffers are first-touched on the GPU's own NUMA node
    n, T = args.envs, args.T
    speed, angle = rt.synthetic_maps(0)
    env = rt.Environment(num_envs=n, seed=SEED + rank * n, maps=(speed, angle), device=dev)   # env shard of this rank

    # rotating inputs: R action buffers + R trajectory buffers, footprint > L2 (126 MB); the same numpy-generated workload as the
    # CPU arm's (make_workload), uploaded before the timed region
    per_buf = T * 2 * n * 4
    R = max(2, int(np.ceil(160e6 / per_buf)) + 1)
    starts_np, acts_np = make_workload(rank, n, T, R)
    env.robot_state = torch.from_numpy(starts_np).to(dev)
    acts = [torch.from_numpy(a).to(dev) for a in acts_np]
    L = rt._lib.lib()
    trajs = [torch.empty((T, 2, n), dtype=torch.float32, device=dev) for _ in range(R)]
    stream = torch.cuda.current_stream(dev)
    sp = rt._lib.stream_ptr(dev)
    LPS = args.launches_per_step

    def one_step(k):
        for j in range(LPS):
            q = (k * LPS + j) % R
            rt._lib.check(L.rtd3_env_rollout(env._handle, rt._lib.ptr(env._state[0]), rt._lib.ptr(env._state[1]),
                                             rt._lib.ptr(acts[q]), rt._lib.ptr(trajs[q]), n, T, sp))

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank)
    sampler.start()

    for k in range(args.warmup):
        one_step(k)
    barrier()
    rt._lib.launch_count_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.in_region = True
    e0.record(stream)
    for k in range(args.steps):
        one_step(args.warmup + k)
    e1.record(stream)
    barrier()
    launches = rt._lib.launch_count()
    if args.dump_outputs and rank == 0:
        last = ((args.warmup + args.steps) * LPS - 1) % R            # trajectory buffer of the last launch of the last step
        dump_outputs(args.dump_outputs, env._state, trajs[last])
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    env_steps_total = float(n) * T * args.steps * LPS * world
    value = env_steps_total / (ms * 1e-3)

    # ---- e2e: host action buffers -> public API -> host trajectory, copies inside the timed region
    h_act = [torch.from_numpy(acts_np[j % R].copy()).pin_memory() for j in range(2)]      # the workload's actions, in pinned host memory
    h_traj = [torch.empty((T, 2, n), dtype=torch.float32).pin_memory() for _ in range(2)]
    e2e_steps = args.steps
    EPS = E2E_CALLS_PER_STEP

    def e2e_step(k):
        # the public host-buffer API: pinned actions in, pinned trajectory out, copies pipelined with the kernel inside the call
        for j in range(EPS):
            env.rollout_host(h_act[(k + j) % 2], h_traj[(k + j) % 2])

    for k in range(3):
        e2e_step(k)
    barrier()
    e0.record(stream)
    for k in range(e2e_steps):
        e2e_step(k)
    e1.record(stream)
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = float(n) * T * e2e_steps * EPS * world / (e2e_ms * 1e-3)

    # ---- configs[4]: envs 1 k ... 1 M per GPU x {single-step kernel (24 B/env-step), T-step rollout kernel (16 B/env-step)} on EVERY
    # rank (weak scaling: the same sizes per GPU, MAX time over the ranks, aggregate env-steps/s), plus the HBM-sized points
    extra = {}
    if not args.no_sweep:
        def timed(go, reps, warm=3):
            for k in range(warm):
                go(k)
            barrier()
            e0.record(stream)
            for k in range(reps):
                go(k)
            e1.record(stream)
            barrier()
            t = torch.tensor([e0.elapsed_time(e1) * 1e3 / reps], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t[0])
        cpu_rate = cpu["value"] if cpu else None
        sweep = []
        for big in (1 << 10, 1 << 12, 1 << 14, 1 << 16, 1 << 18, 1 << 20, 1 << 22, 1 << 24):
            bx = [torch.rand((2, big), device=dev) * 98 for _ in range(3)]          # 3 rotating sets: > L2 at 16M
            ba = [torch.rand((2, big), device=dev) * 15 - 7.5 for _ in range(3)]
            for variant, name in ((1, "smem"), (2, "ldg")):
                if big < (1 << 20) and variant == 1:
                    continue                                                        # (the staged table only pays at HBM-sized batches)
                def go(k):
                    rt._lib.check(L.rtd3_env_step(env._handle, rt._lib.ptr(bx[k % 3][0]), rt._lib.ptr(bx[k % 3][1]),
                                                  rt._lib.ptr(ba[k % 3][0]), rt._lib.ptr(ba[k % 3][1]), big, variant, sp))
                us = timed(go, 30)
                gbs = big * STEP_BYTES_PER_ENV_STEP / (us * 1e-6) / 1e9
                sweep.append({"kernel": "env_step_kernel/" + name, "envs_per_gpu": big, "n_gpus": world, "us": round(us, 2),
                              "env_steps_per_sec": big * world / (us * 1e-6), "GB/s_per_gpu": round(gbs, 1), "frac": round(gbs / hbm_peak, 3),
                              "cpu_port_env_steps_per_sec": cpu_rate})
            del bx, ba
        extra["step_kernel_sweep"] = sweep
        # the T-step rollout kernel (16 B per env-step: action in, state out)
        rsweep = []
        for big, Tb in ((1 << 10, 1000), (1 << 12, 1000), (1 << 14, 1000), (1 << 16, 256), (1 << 18, 128), (1 << 20, 64), (1 << 22, 16)):
            envb = rt.Environment(num_envs=big, seed=5 + rank, maps=(speed, angle), device=dev)
            envb.reset()
            ab = [torch.rand((Tb, 2, big), device=dev) * 15 - 7.5 for _ in range(2)]
            tb = torch.empty((Tb, 2, big), dtype=torch.float32, device=dev)
            def go(k):
                rt._lib.check(L.rtd3_env_rollout(envb._handle, rt._lib.ptr(envb._state[0]), rt._lib.ptr(envb._state[1]),
                                                 rt._lib.ptr(ab[k % 2]), rt._lib.ptr(tb), big, Tb, sp))
            us = timed(go, 10, warm=2)
            gbs = big * Tb * ROLL_BYTES_PER_ENV_STEP / (us * 1e-6) / 1e9
            rsweep.append({"kernel": "env_rollout (auto variant)", "envs_per_gpu": big, "n_gpus": world, "steps": Tb, "us": round(us, 1),
                           "env_steps_per_sec": big * Tb * world / (us * 1e-6), "GB/s_per_gpu": round(gbs, 1), "frac": round(gbs / hbm_peak, 3),
                           "cpu_port_env_steps_per_sec": cpu_rate})
            del envb, ab, tb
        extra["rollout_kernel_sweep"] = rsweep
    td3_rows = None if args.no_td3 else bench_td3(rt, torch, dev, world, rank, cpu=not args.no_cpu)
    fwd_rows = None if (args.no_td3 or rank != 0 or world > 1) else bench_forward(rt, torch, dev)
    loop_row = None if args.no_loop else bench_full_loop(rt, torch, dev, world, rank)
    single_row = bench_single_env(rt, torch, dev) if (world == 1 and not args.no_loop) else None
    sampler.in_region = False
    sampler.stop()

    if rank == 0:
        us_per_launch = ms * 1e3 / (args.steps * LPS)
        alg_bytes = float(n) * T * ROLL_BYTES_PER_ENV_STEP
        achieved = alg_bytes / (us_per_launch * 1e-6) / 1e9
        line = {
            "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD if (n == ENVS and T == T_STEPS) else "batched dynamics rollout: %d envs x %d steps per GPU" % (n, T),
                       "envs_per_gpu": n, "rollout_steps": T, "rollouts_per_bench_step": LPS,
                       "kernel": "env_rollout_pair_kernel<traj> (TMA tiles, chain + helper warp per 32 envs)",
                       "l2": "inputs rotate over %d action + %d trajectory buffers (%.0f MB > 126 MB L2)" % (R, R, 2 * R * per_buf / 1e6)},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                         "traffic": None, "peak_kind": peak_kind,
                         "traffic_note": "not measurable inside this process; the ncu capture of this kernel (profiles/r1_ncu_summaries.md) read 32.9 MB + wrote 0.6 MB of DRAM per launch against 65.5 MB algorithmic (the trajectory is still in L2 at kernel end)",
                         "note": "%d B per env-step (action in 8 B, state out 8 B; state lives in registers) x %d env-steps per launch; "
                                 "4096 envs = 128 chain warps (+128 helper warps) on 148 SMs: one dependent chain per SM, so this config is latency-bound (see step_kernel_sweep for HBM-sized batches)"
                                 % (ROLL_BYTES_PER_ENV_STEP, n * T)},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "env-steps/s",
                    "h2d_bytes_per_step": per_buf * EPS, "d2h_bytes_per_step": per_buf * EPS, "calls_per_step": EPS,
                    "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
                    "path": "Environment.rollout_host on pinned host buffers (rtd3_env_rollout_host): 8 time slices, the copy engine stages "
                            "the actions of slice c+1 in HBM while the rollout kernel runs slice c and writes its trajectory tiles to host "
                            "memory over PCIe (TMA stores), the pipeline replayed as one CUDA graph per call; raw cudaMemcpy of both "
                            "directions run concurrently takes 0.70 ms for these bytes"},
            "gpu_launches": launches,
            "clocks": sampler.summary(),
        }
        line.update(extra)
        if td3_rows is not None:
            line["td3"] = td3_rows
        if fwd_rows is not None:
            line["actor_forward"] = fwd_rows
        if loop_row is not None:
            line["full_loop"] = loop_row
        if single_row is not None:
            line["single_env_loop"] = single_row
        if world > 1:
            flags = [r.get("replicas_identical") for r in (td3_rows or []) + (loop_row or []) if "replicas_identical" in r]
            line["replicas_identical"] = bool(flags) and all(flags)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_RESULT_FD = None


def emit(line):
    """The one JSON line of the contract, on the real stdout (see main)."""
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_RESULT_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--launches-per-step", type=int, default=LAUNCHES_PER_STEP)
    ap.add_argument("--envs", type=int, default=ENVS)
    ap.add_argument("--T", type=int, default=T_STEPS)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-td3", action="store_true")
    ap.add_argument("--no-loop", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the final state and trajectory of the last rollout as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to stdout on the
    # first communicator): point fd 1 at stderr for the whole run and keep the real stdout for the result line only.
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
