"""Checkpoint and resume: the whole state of a training run, saved so that a resumed run is the same run.

`state_dict()` / `load_state_dict(sd)` of `ReplayBuffer`, `TD3`, `Environment`, `Robot`, `BatchedTrainer` and `DriverLoop` are built
here; `save_checkpoint(path, obj)` / `load_checkpoint(path, obj)` write and read them as files.

A state dict is a plain dict: "meta" (class, format version, configuration), "tensors" (CPU tensors keyed by the attribute path of
the object's own tensor: "_state", "_bank.mt", "_env_demo.sets", ...), "host" (Python values) and the state dicts of the objects it
contains.  Loading goes into an existing object of the same configuration: every check runs first (ValueError, nothing written),
then tensors are copied in place, so CUDA graphs the objects have captured stay valid.  What is not stored - data derived from the
stored state and rebuilt on load, scratch and process-local state - is listed per class in NOT_SAVED.

Each `*_state(obj, take)` is the one definition of what is stored: it runs the guards, synchronises, reads the host values and
applies `take` to every stored tensor.  A synchronous save takes CPU copies (`_host`).  A background save
(`save_checkpoint(..., background=True)`) collects the live tensors (`_live`), stages them in device memory with stream-ordered
copies (`_stage`) and returns; a writer thread copies the staging to pinned host memory on a side stream (`_pinned`), frees it and
writes the file.

RNG state is part of the run: every MT19937 bank, the Philox offsets and counters, and - for objects that draw from numpy's global
stream (a single env or robot without a seed) - numpy's global state, which `load_state_dict` RESTORES (a process-wide side effect,
as the reference draws everything from that stream).  With `noise="randn"` the trainer saves and restores torch's CUDA generator.
"""
import atexit
import json
import os
import tempfile
import threading
import weakref

import numpy as np
import torch

from . import _lib

FORMAT = "rtd3_b200 checkpoint"
FORMAT_VERSION = 1

# Tensor attributes (paths as in the state dicts' "tensors") that a state dict does not hold, with the reason.  A prefix covers
# everything below it.  tests/test_checkpoint_gpu.py fails for a tensor attribute that is neither stored nor listed here.
NOT_SAVED = {
    "ReplayBuffer": {"_scratch": "sampler scratch"},
    "TD3": {"params_t": "rebuilt: transposed weights (rtd3_td3_sync_transposed)",
            "params_u": "rebuilt: tensor-core operand copies (rtd3_tc_sync_weights)",
            "params_h": "rebuilt: fp16 weight copies (rtd3_tc_sync_weights_f16)",
            "grads": "scratch: written by every step before it is read", "_scratch": "row scratch", "_scratch_retired": "row scratch",
            "_graphs": "captured update graphs and their buffers",
            "_grads_sum": "peer-memory exchange: process-local", "_p2p": "peer-memory receive areas, flags and seq: process-local"},
    "Environment": {"_speed_dev": "stored under this name unless map_seeds rebuild the bank", "_angle_dev": "as _speed_dev",
                    "_cem": "planner scratch", "_pipe_buf": "host-rollout staging"},
    "Robot": {"goal_state": "view of _goal", "_demo_dev": "rebuilt from demonstration_states",
              "_demo_cells": "rebuilt: candidate lists (rtd3_demo_lists)", "_demo_list": "rebuilt: candidate lists (rtd3_demo_lists)",
              "_env_demo.sorted": "rebuilt: per-env grids (rtd3_robot_demo_grids)", "_env_demo.cells": "rebuilt with _env_demo.sorted",
              "_snap": "folded into host['snap'] at the save", "_eval_graphs": "captured evaluation graphs", "_eval_work": "evaluation scratch"},
    "BatchedTrainer": {"_types": "alias of robot._type"},
    "DriverLoop": {},
}

_BANK = ("mt", "pos", "has_gauss", "gauss")
_REPLAY = ("s", "a", "r", "s2", "notdone", "_total_dev") + tuple("_bank." + k for k in _BANK)
_TD3 = ("params", "adam_m", "adam_v", "steps", "beta_pows", "_noise_counter")
_ENV = ("_state", "_state64", "_goal", "_region") + tuple("_bank." + k for k in _BANK)
_ROBOT = ("_goal", "_num_episodes", "_noise_scale", "_path_length", "_plan_index", "_hist", "_hist_count", "_hist_head", "_goal_reached",
          "_demo_flag", "_stuck_flag", "_type", "_update", "_any_update", "_reward", "_reward64", "_done", "_base", "_action", "_action64"
          ) + tuple("_bank." + k for k in _BANK)
_TRAINER = ("steps_bought", "resets_bought", "_tick_counter", "_prev", "_z")
_SCHEDULER = ("mode", "demos_bought", "test_ticks", "test_best_distance", "test_success", "penalty")
_LOOP_HOST = ("mode", "demos_bought", "resets_bought", "steps_bought", "test_ticks", "test_best_distance", "penalty", "success", "finished",
              "ticks", "tick_seconds", "test_timeout_ticks", "last_action_type")
NETWORKS = ("actor_network", "critic_network_1", "critic_network_2", "target_actor", "target_critic_network_1", "target_critic_network_2")


# ---------------------------------------------------------------------------------------------------------------- helpers
def _get(obj, path):
    for part in path.split("."):
        obj = obj[part] if isinstance(obj, dict) else getattr(obj, part)
    return obj


def _host(t):
    """A CPU copy of a tensor (None stays None)."""
    if t is None:
        return None
    return t.detach().cpu() if t.is_cuda else t.detach().clone()


def _live(t):
    """The tensor itself: a background save collects the state with this `take`, then stages the tensors (`_stage`)."""
    return None if t is None else t.detach()


def _stage(t):
    """A copy of a tensor on its own device: stream-ordered on the current stream for a device tensor."""
    return t.clone()


def _pinned(t):
    """A pinned host copy of a device tensor, enqueued on the current stream (a background save's writer thread)."""
    if not t.is_cuda:
        return t
    return torch.empty_like(t, device="cpu", pin_memory=True).copy_(t, non_blocking=True)


def _map(sd, fn):
    """`sd` with `fn` applied to every tensor in it."""
    if isinstance(sd, torch.Tensor):
        return fn(sd)
    if isinstance(sd, dict):
        return {k: _map(v, fn) for k, v in sd.items()}
    if isinstance(sd, (list, tuple)):
        return type(sd)(_map(v, fn) for v in sd)
    return sd


def _tensors(obj, names, take=_host):
    return {k: take(_get(obj, k)) for k in names}


def _check_tensor(t, dtype, shape, what):
    if not isinstance(t, torch.Tensor):
        raise ValueError("checkpoint: %s is missing or not a tensor" % what)
    if t.dtype != dtype or tuple(t.shape) != tuple(shape):
        raise ValueError("checkpoint: %s is %s %s, expected %s %s" % (what, t.dtype, list(t.shape), dtype, list(shape)))


def _check_like(sd, obj, names, cls):
    """Every named tensor is present with the live tensor's dtype and shape."""
    tensors = _section(sd, "tensors", cls)
    for k in names:
        live = _get(obj, k)
        _check_tensor(tensors.get(k), live.dtype, live.shape, "%s tensor %r" % (cls, k))


def _section(sd, key, cls):
    if not isinstance(sd, dict) or not isinstance(sd.get(key), dict):
        raise ValueError("checkpoint: %s state has no %r section" % (cls, key))
    return sd[key]


def _check_meta(sd, cls, **expect):
    meta = _section(sd, "meta", cls)
    if meta.get("class") != cls:
        raise ValueError("checkpoint: state of a %s, expected a %s" % (meta.get("class"), cls))
    if meta.get("version") != FORMAT_VERSION:
        raise ValueError("checkpoint: format version %r, this build reads %d" % (meta.get("version"), FORMAT_VERSION))
    for k, v in expect.items():
        if meta.get(k) != v:
            raise ValueError("checkpoint: %s %s is %r, the target has %r" % (cls, k, meta.get(k), v))
    _section(sd, "tensors", cls)
    _section(sd, "host", cls)


def _copy_in(obj, tensors, names):
    for k in names:
        _get(obj, k).copy_(tensors[k])


def _numpy_state():
    name, keys, pos, has_gauss, cached = np.random.get_state()
    return {"keys": torch.from_numpy(keys.astype(np.int64)), "pos": int(pos), "has_gauss": int(has_gauss), "gauss": float(cached)}


def _check_numpy_state(st, cls):
    if not isinstance(st, dict):
        raise ValueError("checkpoint: %s state lacks numpy's global stream" % cls)
    _check_tensor(st.get("keys"), torch.int64, (624,), "%s numpy keys" % cls)
    for k, typ in (("pos", int), ("has_gauss", int), ("gauss", float)):
        if not isinstance(st.get(k), typ):
            raise ValueError("checkpoint: %s numpy state field %r is missing" % (cls, k))


def _set_numpy_state(st):
    np.random.set_state(("MT19937", st["keys"].numpy().astype(np.uint32), st["pos"], st["has_gauss"], st["gauss"]))


def _rank_world(td3):
    if td3.world == 1:
        return 0, 1
    import torch.distributed as dist
    return dist.get_rank(td3.process_group), td3.world


def _quiescent(device):
    if torch.cuda.is_current_stream_capturing():
        raise RuntimeError("cannot save a checkpoint inside a CUDA graph capture")
    torch.cuda.synchronize(device)


# ---------------------------------------------------------------------------------------------------------------- ReplayBuffer
def replay_state(rb, take=_host):
    if rb._in_session:
        raise RuntimeError("cannot save a ReplayBuffer inside an open sampling session")
    _quiescent(rb.device)
    host = {"sampler": rb.sampler, "philox_seed": rb._philox_seed, "philox_offset": rb._philox_offset,
            "numpy": _numpy_state() if rb._numpy_global else None}
    return {"meta": {"class": "ReplayBuffer", "version": FORMAT_VERSION, "capacity": rb.capacity, "numpy_global": rb._numpy_global},
            "tensors": _tensors(rb, _REPLAY, take), "host": host}


def replay_plan(rb, sd):
    _check_meta(sd, "ReplayBuffer", capacity=rb.capacity, numpy_global=rb._numpy_global)
    _check_like(sd, rb, _REPLAY, "ReplayBuffer")
    t, h = sd["tensors"], sd["host"]
    if h.get("sampler") not in ("mt19937", "philox") or not isinstance(h.get("philox_seed"), int) or not isinstance(h.get("philox_offset"), int):
        raise ValueError("checkpoint: ReplayBuffer sampler state is missing")
    if rb._numpy_global:
        _check_numpy_state(h.get("numpy"), "ReplayBuffer")

    def apply():
        _copy_in(rb, t, _REPLAY)
        rb._total_host, rb._host_stale = int(t["_total_dev"][0]), False
        rb.sampler, rb._philox_seed, rb._philox_offset = h["sampler"], h["philox_seed"], h["philox_offset"]
        if rb._numpy_global:
            _set_numpy_state(h["numpy"])
    return [apply]


# ---------------------------------------------------------------------------------------------------------------- TD3
def td3_state(td3, take=_host):
    _quiescent(td3.device)
    rank, world = _rank_world(td3)
    last = None if td3.last_losses is None else [take(x) for x in td3.last_losses]
    return {"meta": {"class": "TD3", "version": FORMAT_VERSION, "hidden": td3.hidden, "layers": td3.layers, "rank": rank, "world": world},
            "tensors": _tensors(td3, _TD3, take),
            "host": {"noise_steps": td3._noise_steps, "noise_seed": td3.noise_seed, "last_losses": last}}


def _rebuild_weights(td3):
    """The derived weight copies from the (new) arena, with the kernels that build them during training."""
    td3.sync_transposed(force=True)
    if td3.params_u is not None:
        td3._sync_chunk_major()
    if td3.params_h is not None:
        td3._sync_half(force=True)


def td3_plan(td3, sd):
    rank, world = _rank_world(td3)
    _check_meta(sd, "TD3", hidden=td3.hidden, layers=td3.layers, rank=rank, world=world)
    _check_like(sd, td3, _TD3, "TD3")
    t, h = sd["tensors"], sd["host"]
    if not isinstance(h.get("noise_steps"), int) or not isinstance(h.get("noise_seed"), int):
        raise ValueError("checkpoint: TD3 noise counter is missing")
    last = h.get("last_losses")
    if last is not None and not (isinstance(last, list) and len(last) == 2 and all(isinstance(x, torch.Tensor) for x in last)):
        raise ValueError("checkpoint: TD3 last_losses must be two tensors")

    def apply():
        _copy_in(td3, t, _TD3)
        td3._noise_steps, td3.noise_seed = h["noise_steps"], h["noise_seed"]
        td3.last_losses = None if last is None else tuple(x.to(td3.device) for x in last)
        _rebuild_weights(td3)
    return [apply]


def export_networks(td3):
    """The six networks as `nn.Module` state dicts: {attribute name: {"layer_1.weight": ..., "output_layer.bias": ...}}, CPU float32."""
    torch.cuda.synchronize(td3.device)
    out = {}
    for k, name in enumerate(NETWORKS):
        net = getattr(td3, name)
        names = ["layer_%d" % (i + 1) for i in range(len(net._layers) - 1)] + ["output_layer"]
        out[name] = {}
        for lname, lv in zip(names, net._layers):
            out[name][lname + ".weight"] = lv.weight.detach().cpu().clone()
            out[name][lname + ".bias"] = lv.bias.detach().cpu().clone()
    return out


def import_networks(td3, d):
    """Inverse of `export_networks`: every network and layer is checked first (ValueError, nothing written)."""
    if not isinstance(d, dict):
        raise ValueError("import_networks takes the dict export_networks returns")
    todo = []
    for name in NETWORKS:
        net = getattr(td3, name)
        sd = d.get(name)
        if not isinstance(sd, dict):
            raise ValueError("import_networks: network %r is missing" % name)
        names = ["layer_%d" % (i + 1) for i in range(len(net._layers) - 1)] + ["output_layer"]
        if set(sd) != {n + s for n in names for s in (".weight", ".bias")}:
            raise ValueError("import_networks: network %r has keys %s" % (name, sorted(sd)))
        for lname, lv in zip(names, net._layers):
            for suffix, live in ((".weight", lv.weight), (".bias", lv.bias)):
                v = sd[lname + suffix]
                _check_tensor(v, torch.float32, live.shape, "%s.%s%s" % (name, lname, suffix))
                todo.append((live, v))
    for live, v in todo:
        live.copy_(v)
    _rebuild_weights(td3)


# ---------------------------------------------------------------------------------------------------------------- Environment
def env_state(env, take=_host):
    _quiescent(env.device)
    names = _ENV + (("_map_seeds",) if env._map_seeds is not None else ("_speed_dev", "_angle_dev"))
    t = _tensors(env, names, take)
    t["_map_index"] = take(env._map_index)
    host = {"numpy": _numpy_state() if env._numpy_global else None,
            "state_np": None if env._state_np is None else torch.from_numpy(np.array(env._state_np, dtype=np.float64))}
    return {"meta": {"class": "Environment", "version": FORMAT_VERSION, "num_envs": env.num_envs, "num_maps": env.num_maps,
                     "numpy_global": env._numpy_global},
            "tensors": t, "host": host}


def env_plan(env, sd):
    from .environment import _checked_seeds, _perlin_maps_device
    n = env.num_envs
    _check_meta(sd, "Environment", num_envs=n, numpy_global=env._numpy_global)
    _check_like(sd, env, _ENV, "Environment")
    t, h = sd["tensors"], sd["host"]
    W = 100
    if t.get("_map_seeds") is not None:
        seeds = _checked_seeds(t["_map_seeds"])
        K = seeds.shape[0]
        speed = angle = None
    else:
        speed, angle = t.get("_speed_dev"), t.get("_angle_dev")
        if not isinstance(speed, torch.Tensor) or speed.dim() not in (2, 3):
            raise ValueError("checkpoint: Environment maps are missing")
        K = 1 if speed.dim() == 2 else speed.shape[0]
        for name, m in (("speed", speed), ("angle", angle)):
            _check_tensor(m, torch.float32, speed.shape if speed.dim() == 2 else (K, W, W), "Environment map %s" % name)
        if tuple(speed.shape[-2:]) != (W, W) or K < 1:
            raise ValueError("checkpoint: Environment maps must be [100,100] or [K,100,100]")
    index = t.get("_map_index")
    if index is not None:
        _check_tensor(index, torch.int32, (n,), "Environment map index")
        if n and (int(index.min()) < 0 or int(index.max()) >= K):
            raise ValueError("checkpoint: Environment map index outside [0, %d)" % K)
    if env._numpy_global:
        _check_numpy_state(h.get("numpy"), "Environment")
    state_np = h.get("state_np")
    if state_np is not None:
        _check_tensor(state_np, torch.float64, (2,), "Environment host state")

    def apply():
        _copy_in(env, t, _ENV)
        # the map tables go back in place (same K: same bank and index addresses, so captured graphs stay valid)
        if speed is None:
            env._install_maps(*_perlin_maps_device(seeds, env.device), index, seeds=seeds)
        else:
            env._install_maps(speed, angle, index)
        env._state_np = None if state_np is None else state_np.numpy().copy()
        if env._numpy_global:
            _set_numpy_state(h["numpy"])
    return [apply]


# ---------------------------------------------------------------------------------------------------------------- Robot
def robot_state(robot, take=_host):
    _quiescent(robot.device)
    t = _tensors(robot, _ROBOT, take)
    d = robot._env_demo
    env_demo = None
    if d is not None:
        k = int(d["count"].max()) if robot.num_envs else 0
        t["_env_demo.sets"] = take(d["sets"][:, :k])
        t["_env_demo.count"] = take(d["count"])
        env_demo = {"cap": int(d["cap"]), "demos": int(d["demos"])}
    arr = lambda rows: None if not rows else torch.from_numpy(np.asarray([np.asarray(r, dtype=np.float64) for r in rows], dtype=np.float64))
    snap = None
    if robot._snap is not None:
        s = robot._snap
        snap = {"seen": int(s["seen"]), "pending": s["event"] is not None, "value": int(s["host"][0]) if s["event"] is not None else 0}
    host = {"num_updates": robot.num_updates, "episodes_per_update": int(robot.episodes_per_update), "env_demo": env_demo,
            "demonstration_states": arr(robot.demonstration_states), "demonstration_actions": arr(robot.demonstration_actions),
            "snap": snap, "numpy": _numpy_state() if robot._numpy_global else None}
    return {"meta": {"class": "Robot", "version": FORMAT_VERSION, "num_envs": robot.num_envs, "batched": robot.batched,
                     "numpy_global": robot._numpy_global},
            "tensors": t, "host": host, "memory": replay_state(robot.memory, take), "td3_agent": td3_state(robot.td3_agent, take)}


def robot_plan(robot, sd):
    n = robot.num_envs
    _check_meta(sd, "Robot", num_envs=n, batched=robot.batched, numpy_global=robot._numpy_global)
    _check_like(sd, robot, _ROBOT, "Robot")
    plan = replay_plan(robot.memory, sd.get("memory")) + td3_plan(robot.td3_agent, sd.get("td3_agent"))
    t, h = sd["tensors"], sd["host"]
    if not isinstance(h.get("num_updates"), int) or not isinstance(h.get("episodes_per_update"), int):
        raise ValueError("checkpoint: Robot update counters are missing")
    for k in ("demonstration_states", "demonstration_actions"):
        v = h.get(k)
        if v is not None and (not isinstance(v, torch.Tensor) or v.dtype != torch.float64 or v.dim() != 2 or v.shape[1] != 2):
            raise ValueError("checkpoint: Robot %s must be float64 [M,2]" % k)
    ed = h.get("env_demo")
    if ed is not None:
        if not isinstance(ed.get("cap"), int) or ed["cap"] < 1 or not isinstance(ed.get("demos"), int):
            raise ValueError("checkpoint: Robot per-env demonstration capacity is missing")
        _check_tensor(t.get("_env_demo.count"), torch.int32, (n,), "Robot _env_demo.count")
        sets = t.get("_env_demo.sets")
        if not isinstance(sets, torch.Tensor) or sets.dim() != 3 or sets.shape[1] > ed["cap"]:
            raise ValueError("checkpoint: Robot _env_demo.sets must be [N,k,2] with k <= cap")
        _check_tensor(sets, torch.float64, (n, sets.shape[1], 2), "Robot _env_demo.sets")
        if n and int(t["_env_demo.count"].max()) > sets.shape[1]:
            raise ValueError("checkpoint: Robot _env_demo.count exceeds the stored sets")
    snap = h.get("snap")
    if snap is not None and not all(isinstance(snap.get(k), int) for k in ("seen", "value")):
        raise ValueError("checkpoint: Robot update snapshot is malformed")
    if robot._numpy_global:
        _check_numpy_state(h.get("numpy"), "Robot")

    def apply():
        _copy_in(robot, t, _ROBOT)
        if not robot.batched:
            robot.goal_state = t["_goal"][:, 0].numpy().copy()
        robot.num_updates, robot.episodes_per_update = h["num_updates"], h["episodes_per_update"]
        rows = lambda v: [] if v is None else list(v.numpy().copy())
        new = rows(h["demonstration_states"])
        old = np.asarray(robot.demonstration_states, dtype=np.float64)
        robot.demonstration_actions = rows(h["demonstration_actions"])
        if not (len(new) == len(old) and np.array_equal(np.asarray(new, dtype=np.float64).reshape(old.shape), old)):
            robot.demonstration_states = new                     # a different shared set: re-uploaded (its graphs are re-captured)
            robot._upload_demos()
        else:
            robot.demonstration_states = new
        _load_env_demo(robot, ed, t)
        if snap is None:
            robot._snap = None
        else:
            robot._snap = {"dev": torch.zeros(1, dtype=torch.int64, device=robot.device),
                           "host": torch.tensor([snap["value"]], dtype=torch.int64).pin_memory(), "event": None, "seen": snap["seen"]}
            if snap["pending"]:                                   # the next maybe_update_async takes the decision the original would
                robot._snap["event"] = torch.cuda.Event()
                robot._snap["event"].record(torch.cuda.current_stream(robot.device))
        if robot._numpy_global:
            _set_numpy_state(h["numpy"])
    return plan + [apply]


def _load_env_demo(robot, ed, t):
    """Per-env sets back in place (reallocated only for another capacity) and their search grids rebuilt."""
    if ed is None:
        robot._env_demo = None
        return
    n, cap, dev = robot.num_envs, ed["cap"], robot.device
    d = robot._env_demo
    if d is None or d["cap"] != cap:
        f64 = lambda: torch.zeros((n, cap, 2), dtype=torch.float64, device=dev)
        d = robot._env_demo = {"cap": cap, "sets": f64(), "sorted": f64(), "count": torch.zeros((n,), dtype=torch.int32, device=dev),
                               "cells": torch.zeros((n, 626), dtype=torch.int32, device=dev)}
    d["demos"] = ed["demos"]
    sets = t["_env_demo.sets"]
    d["sets"].zero_()
    d["sets"][:, :sets.shape[1]].copy_(sets)
    d["count"].copy_(t["_env_demo.count"])
    d["sorted"].zero_()
    _lib.check(_lib.lib().rtd3_robot_demo_grids(_lib.ptr(d["sets"]), _lib.ptr(d["count"]), cap, n, _lib.ptr(d["sorted"]), _lib.ptr(d["cells"]),
                                                _lib.stream_ptr(dev)), "robot_demo_grids")


# ---------------------------------------------------------------------------------------------------------------- BatchedTrainer
def trainer_state(tr, take=_host):
    _quiescent(tr.device)
    rank, world = _rank_world(tr.robot.td3_agent)
    names = _TRAINER + (_SCHEDULER if tr.scheduler else ())
    host = {"ticks": tr.ticks, "philox_seed": tr.philox_seed,
            "cuda_rng": torch.cuda.get_rng_state(tr.device) if tr.noise == "randn" else None}
    return {"meta": {"class": "BatchedTrainer", "version": FORMAT_VERSION, "num_envs": tr.n, "noise": tr.noise, "scheduler": tr.scheduler,
                     "rank": rank, "world": world},
            "tensors": _tensors(tr, names, take), "host": host, "env": env_state(tr.env, take), "robot": robot_state(tr.robot, take)}


def trainer_plan(tr, sd):
    rank, world = _rank_world(tr.robot.td3_agent)
    _check_meta(sd, "BatchedTrainer", num_envs=tr.n, noise=tr.noise, scheduler=tr.scheduler, rank=rank, world=world)
    names = _TRAINER + (_SCHEDULER if tr.scheduler else ())
    _check_like(sd, tr, names, "BatchedTrainer")
    plan = env_plan(tr.env, sd.get("env")) + robot_plan(tr.robot, sd.get("robot"))
    t, h = sd["tensors"], sd["host"]
    if not isinstance(h.get("ticks"), int) or not isinstance(h.get("philox_seed"), int):
        raise ValueError("checkpoint: BatchedTrainer tick counters are missing")
    if tr.noise == "randn" and not isinstance(h.get("cuda_rng"), torch.Tensor):
        raise ValueError("checkpoint: BatchedTrainer with noise='randn' needs torch's CUDA generator state")

    def apply():
        _copy_in(tr, t, names)
        tr.ticks, tr.philox_seed = h["ticks"], h["philox_seed"]
        if hasattr(tr, "_types"):
            tr._types = tr.robot._type
        if tr.noise == "randn":
            torch.cuda.set_rng_state(h["cuda_rng"], tr.device)
    return plan + [apply]


# ---------------------------------------------------------------------------------------------------------------- DriverLoop
def loop_state(loop, take=_host):
    host = {k: float(v) if isinstance(v, float) else v for k, v in ((k, getattr(loop, k)) for k in _LOOP_HOST)}   # numpy floats -> float
    host["state"] = torch.from_numpy(np.array(loop.state))
    return {"meta": {"class": "DriverLoop", "version": FORMAT_VERSION, "num_envs": loop.environment.num_envs},
            "tensors": {}, "host": host, "env": env_state(loop.environment, take), "robot": robot_state(loop.robot, take)}


def loop_plan(loop, sd):
    _check_meta(sd, "DriverLoop", num_envs=loop.environment.num_envs)
    plan = env_plan(loop.environment, sd.get("env")) + robot_plan(loop.robot, sd.get("robot"))
    h = sd["host"]
    missing = [k for k in _LOOP_HOST + ("state",) if k not in h]
    if missing or h["mode"] not in ("training", "testing"):
        raise ValueError("checkpoint: DriverLoop state lacks %s" % (missing or ["a valid mode"]))

    def apply():
        for k in _LOOP_HOST:
            setattr(loop, k, h[k])
        loop.state = h["state"].numpy().copy()
    return plan + [apply]


# ---------------------------------------------------------------------------------------------------------------- dispatch and files
def _kind(obj):
    from .environment import Environment
    from .learner import TD3, ReplayBuffer
    from .robot import Robot
    from .trainer import BatchedTrainer, DriverLoop
    for cls, save, plan in ((ReplayBuffer, replay_state, replay_plan), (TD3, td3_state, td3_plan), (Environment, env_state, env_plan),
                            (Robot, robot_state, robot_plan), (BatchedTrainer, trainer_state, trainer_plan), (DriverLoop, loop_state, loop_plan)):
        if isinstance(obj, cls):
            return cls.__name__, save, plan
    raise TypeError("checkpoints cover ReplayBuffer, TD3, Environment, Robot, BatchedTrainer and DriverLoop, not %s" % type(obj).__name__)


def load_state(obj, sd):
    """Validate `sd` against `obj` as a whole, then write it: a ValueError leaves every tensor of `obj` unchanged."""
    _, _, plan = _kind(obj)
    for step in plan(obj, sd):
        step()
    torch.cuda.synchronize()


def _learner(obj):
    for path in ("robot.td3_agent", "td3_agent"):
        try:
            return _get(obj, path)
        except AttributeError:
            pass
    from .learner import TD3
    return obj if isinstance(obj, TD3) else None


def _summary(obj):
    """The file's plain metadata: what the run is, for a reader of the file (load checks the state dicts' own "meta")."""
    td3 = _learner(obj)
    rank, world = _rank_world(td3) if td3 is not None else (0, 1)
    env = getattr(obj, "env", None) or getattr(obj, "environment", None) or (obj if type(obj).__name__ == "Environment" else None)
    rb = obj if type(obj).__name__ == "ReplayBuffer" else (_get(obj, "robot.memory") if hasattr(obj, "robot") else getattr(obj, "memory", None))
    return {"format": FORMAT, "version": FORMAT_VERSION, "class": type(obj).__name__,
            "num_envs": getattr(obj, "num_envs", None) or getattr(obj, "n", None) or (env.num_envs if env is not None else None),
            "hidden": None if td3 is None else td3.hidden, "layers": None if td3 is None else td3.layers,
            "capacity": None if rb is None else rb.capacity, "num_maps": None if env is None else env.num_maps,
            "rank": rank, "world": world, "noise": getattr(obj, "noise", None)}


def _atomic_save(payload, path):
    """torch.save to a temporary file in the target's directory, then os.replace: an interrupted save leaves `path` as it was."""
    d = os.path.dirname(os.path.abspath(path))
    fd, tmp = tempfile.mkstemp(dir=d, prefix="." + os.path.basename(path) + ".", suffix=".tmp")
    try:
        with os.fdopen(fd, "wb") as f:
            torch.save(payload, f)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, path)
    except BaseException:
        try:
            os.unlink(tmp)
        except OSError:
            pass
        raise


def _read(path):
    payload = torch.load(path, map_location="cpu", weights_only=True)
    meta = payload.get("meta") if isinstance(payload, dict) else None
    if not isinstance(meta, dict) or meta.get("format") != FORMAT:
        raise ValueError("%s is not a checkpoint of this package" % path)
    if meta.get("version") != FORMAT_VERSION:
        raise ValueError("checkpoint %s has format version %r, this build reads %d" % (path, meta.get("version"), FORMAT_VERSION))
    return payload


def _clear_manifest(pg, rank, path):
    """Data parallel, before the rank files are written (collective): rank 0 removes the manifest, so a directory whose save is
    interrupted does not load."""
    import torch.distributed as dist
    manifest = os.path.join(path, "manifest.json")
    if rank == 0:
        os.makedirs(path, exist_ok=True)
        if os.path.exists(manifest):
            os.unlink(manifest)
    dist.barrier(group=pg)


def _write_manifest(pg, rank, world, path, name, num_envs):
    """Data parallel, once every rank file is written (collective): rank 0 writes the manifest."""
    import torch.distributed as dist
    manifest = os.path.join(path, "manifest.json")
    sizes = [None] * world
    dist.all_gather_object(sizes, num_envs, group=pg)
    if rank == 0:
        tmp = manifest + ".tmp"
        with open(tmp, "w") as f:
            json.dump({"format": FORMAT, "version": FORMAT_VERSION, "class": name, "world": world, "num_envs": sizes}, f)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, manifest)
    dist.barrier(group=pg)


def save_checkpoint(path, obj, background=False):
    """Save `obj` (any of the six classes, with everything it contains) to `path`; returns `path`.

    Single process: one file, written atomically.  Data parallel (the learner has a process group of world > 1): collective, `path`
    is a directory; every rank writes `rank{r}.pt` (its env shard, robot, replay shard and learner copy), then rank 0 writes
    `manifest.json` (world, format version, per-rank num_envs).  The manifest is removed before the rank files are written, so a
    directory whose save was interrupted does not load.

    `background=True` returns a `PendingCheckpoint` as soon as the state is snapshot into device memory: the device->host copies
    and the file write run in a writer thread while training continues.  The file is the one a synchronous save at the call would
    write.  Device memory for the stored state is needed twice until the writer has copied it out (RuntimeError, nothing done,
    when `torch.cuda.mem_get_info` reports less free); a second background save of the same object first waits for the first's
    writer.  Data parallel, the call and `PendingCheckpoint.wait()` are collective; the writers never use the process group."""
    name, save, _ = _kind(obj)
    if background:
        return _save_background(path, obj, name, save)
    sd = save(obj)
    payload = {"meta": _summary(obj), "state": sd}
    td3 = _learner(obj)
    rank, world = _rank_world(td3) if td3 is not None else (0, 1)
    if world == 1:
        _atomic_save(payload, path)
        return path
    pg = td3.process_group
    _clear_manifest(pg, rank, path)
    _atomic_save(payload, os.path.join(path, "rank%d.pt" % rank))
    _write_manifest(pg, rank, world, path, name, payload["meta"]["num_envs"])
    return path


# ---------------------------------------------------------------------------------------------------------------- background saves
_PENDING = weakref.WeakKeyDictionary()          # object -> its latest background save
_WRITERS = []                                   # writer threads not yet seen finished


@atexit.register
def _join_writers():
    """A process that exits with a background save pending still finishes the file."""
    for t in list(_WRITERS):
        t.join()


class PendingCheckpoint:
    """A checkpoint being written in the background, returned by `save_checkpoint(path, obj, background=True)`.

    `done()` tells whether this process's writer thread has finished.  `wait()` returns `path` once the file is complete, or
    re-raises the writer's exception (the file at `path` is then as it was).  Data parallel, `wait()` is collective: every rank joins
    its writer, then rank 0 writes the manifest if every rank wrote its file; if any rank failed there is no manifest and every
    rank raises."""

    def __init__(self, path, file, staged, meta, device, event, finish):
        self.path = path
        self._finish, self._error, self._waited = finish, None, False
        self._thread = threading.Thread(target=self._drain, args=(file, staged, meta, device, event), name="rtd3-checkpoint-writer")
        _WRITERS[:] = [t for t in _WRITERS if t.is_alive()] + [self._thread]
        self._thread.start()

    def _drain(self, file, staged, meta, device, event):
        """The writer thread: device->host copies on a side stream once the snapshot is complete, the staging freed, then the file."""
        try:
            with torch.cuda.device(device):
                side = torch.cuda.Stream(device)
                side.wait_event(event)
                try:
                    with torch.cuda.stream(side):
                        state = _map(staged[0], _pinned)
                finally:
                    side.synchronize()
                    staged.clear()                      # the last reference to the device staging
            _atomic_save({"meta": meta, "state": state}, file)
        except BaseException as e:                      # noqa: B036 - handed to wait()
            self._error = e

    def done(self):
        return not self._thread.is_alive()

    def wait(self):
        if not self._waited:
            self._thread.join()
            if self._finish is not None:
                self._error = self._finish(self._error)
            self._waited = True
        if self._error is not None:
            raise self._error
        return self.path


def _save_background(path, obj, name, save):
    """The call of a background save: the synchronous save's guards and host reads, a size check, then device->device copies of
    every stored tensor on the current stream and an event the writer thread waits on."""
    prev = _PENDING.get(obj)
    if prev is not None:
        prev._thread.join()                             # at most one staging copy of an object's state
    live = save(obj, _live)                             # refuses a capture or an open session, synchronises, reads host values
    meta = _summary(obj)
    leaves = []
    _map(live, leaves.append)
    cuda = [t for t in leaves if t.is_cuda]
    device = cuda[0].device
    need = sum(t.numel() * t.element_size() for t in cuda)
    free = torch.cuda.mem_get_info(device)[0]
    td3 = _learner(obj)
    rank, world = _rank_world(td3) if td3 is not None else (0, 1)
    fits = need <= free
    if world > 1:                                       # every rank goes on, or none does
        import torch.distributed as dist
        flag = torch.tensor([int(fits)], dtype=torch.int32, device=td3.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=td3.process_group)
        if fits and not int(flag.item()):
            raise RuntimeError("background checkpoint: another rank lacks the device memory for its snapshot")
    if not fits:
        raise RuntimeError("background checkpoint: the snapshot needs %.2f GB of device memory, %.2f GB are free; save with "
                           "background=False" % (need / 1e9, free / 1e9))
    file, finish = path, None
    if world > 1:
        pg = td3.process_group
        _clear_manifest(pg, rank, path)
        file = os.path.join(path, "rank%d.pt" % rank)

        def finish(error):
            import torch.distributed as dist
            ok = torch.tensor([0 if error else 1], dtype=torch.int32, device=td3.device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=pg)
            if not int(ok.item()):
                return error or RuntimeError("%s: another rank failed to write its checkpoint file" % path)
            _write_manifest(pg, rank, world, path, name, meta["num_envs"])
            return None
    staged = [_map(live, _stage)]
    event = torch.cuda.Event()
    event.record(torch.cuda.current_stream(device))
    pending = _PENDING[obj] = PendingCheckpoint(path, file, staged, meta, device, event, finish)
    return pending


def load_checkpoint(path, obj):
    """Load a checkpoint written by `save_checkpoint` into `obj`, an existing object of the same class and configuration
    (`load_state_dict` semantics: ValueError before anything is written).  Data parallel: collective; the same world size and
    per-rank num_envs are required, and afterwards the learner replicas must be bit-identical (ValueError otherwise)."""
    name, _, plan = _kind(obj)
    td3 = _learner(obj)
    rank, world = _rank_world(td3) if td3 is not None else (0, 1)
    if world == 1:
        if os.path.isdir(path):
            raise ValueError("%s is a data-parallel checkpoint directory; this %s has no process group" % (path, name))
        payload = _read(path)
        if payload["meta"].get("class") != name:
            raise ValueError("checkpoint holds a %s, not a %s" % (payload["meta"].get("class"), name))
        load_state(obj, payload["state"])
        return obj
    import torch.distributed as dist
    from .trainer import replicas_identical
    pg = td3.process_group
    error = None
    try:
        with open(os.path.join(path, "manifest.json")) as f:
            manifest = json.load(f)
        if manifest.get("format") != FORMAT or manifest.get("version") != FORMAT_VERSION or manifest.get("class") != name:
            raise ValueError("%s: manifest of another format, version or class" % path)
        if manifest.get("world") != world:
            raise ValueError("%s was saved by %r ranks, this run has %d (resharding is not supported)" % (path, manifest.get("world"), world))
        payload = _read(os.path.join(path, "rank%d.pt" % rank))
        if manifest["num_envs"][rank] != _summary(obj)["num_envs"]:
            raise ValueError("%s: rank %d saved %r envs" % (path, rank, manifest["num_envs"][rank]))
        steps = plan(obj, payload["state"])
    except (OSError, ValueError, KeyError, IndexError, TypeError) as e:
        error = e
    ok = torch.tensor([0 if error else 1], dtype=torch.int32, device=td3.device)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=pg)          # every rank loads, or none does
    if error is not None:
        raise ValueError(str(error)) from error
    if int(ok.item()) == 0:
        raise ValueError("%s: another rank rejected its part of the checkpoint" % path)
    for step in steps:
        step()
    torch.cuda.synchronize(td3.device)
    if not replicas_identical(td3, pg):
        raise ValueError("%s: the learner replicas differ after loading" % path)
    return obj
