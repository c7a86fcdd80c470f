"""Checkpoint and resume on the B200: a resumed run is the same run.

A resumed run is compared with a FORK of the original: the same objects continuing from the saved point.  Arrays are compared bit
for bit; replay rows and the per-cell contents of the per-env demonstration grids as multisets (masked pushes reserve rows with one
atomicAdd per warp and the grid's counting sort places a cell's states with atomics, so their order varies from run to run)."""
import os
import shutil
import subprocess
import sys
from importlib import import_module

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ck():
    return import_module("residual-td3-robot-navigation_b200.checkpoint")


def _flat(sd, prefix=""):
    """(path, value) of every tensor and plain value of a state dict."""
    if isinstance(sd, dict):
        for k, v in sd.items():
            yield from _flat(v, prefix + str(k) + "/")
    elif isinstance(sd, (list, tuple)):
        for i, v in enumerate(sd):
            yield from _flat(v, prefix + str(i) + "/")
    else:
        yield prefix[:-1], sd


def _rows(sd):
    t = sd["tensors"]
    n = min(int(t["_total_dev"][0]), sd["meta"]["capacity"])
    rows = torch.cat([t["s"][:n], t["a"][:n], t["r"][:n, None], t["s2"][:n], t["notdone"][:n, None]], 1).double().numpy()
    return np.unique(rows, axis=0, return_counts=True)


def assert_same_state(a, b):
    """Every value of two state dicts equal bit for bit, replay rows as multisets."""
    fa, fb = dict(_flat(a)), dict(_flat(b))
    assert fa.keys() == fb.keys()
    ring = {"s", "a", "r", "s2", "notdone"}
    for k, va in fa.items():
        vb = fb[k]
        parts = k.split("/")
        if parts[-2:-1] == ["tensors"] and parts[-1] in ring and "memory" in parts:
            continue
        if isinstance(va, torch.Tensor):
            assert va.dtype == vb.dtype and va.shape == vb.shape, k
            assert torch.equal(va.view(-1).view(torch.uint8) if va.is_floating_point() else va,
                               vb.view(-1).view(torch.uint8) if vb.is_floating_point() else vb), k
        else:
            assert va == vb, (k, va, vb)
    for path in {k.rsplit("/tensors/", 1)[0] for k in fa if k.endswith("/tensors/_total_dev")}:
        sub_a, sub_b = a, b
        for p in path.split("/"):
            if p:
                sub_a, sub_b = sub_a[p], sub_b[p]
        ra, rb = _rows(sub_a), _rows(sub_b)
        assert np.array_equal(ra[0], rb[0]) and np.array_equal(ra[1], rb[1]), path


def grid_key(robot):
    """The per-env grids as (cells, states sorted within each cell) - exact cells, cell contents as multisets."""
    d = robot._env_demo
    if d is None:
        return None
    cells, pts, count = d["cells"], d["sorted"], d["count"]
    pos = torch.arange(pts.shape[1], device=pts.device).expand(pts.shape[0], -1).contiguous()
    cell = torch.searchsorted(cells.contiguous(), pos, right=True) - 1
    cell = torch.where(pos < count[:, None].long(), cell, torch.full_like(cell, 1 << 20))
    order = torch.arange(pts.shape[1], device=pts.device).expand_as(pos)
    for key in (pts[..., 1], pts[..., 0], cell):                    # lexicographic (cell, x, y) by stable sorts, last key first
        k = torch.gather(key, 1, order)
        order = torch.gather(order, 1, torch.sort(k, dim=1, stable=True)[1])
    srt = torch.gather(pts, 1, order[..., None].expand(-1, -1, 2))
    srt = torch.where((torch.gather(cell, 1, order) < (1 << 20))[..., None], srt, torch.zeros_like(srt))
    return cells.cpu(), srt.cpu()


def assert_same_grids(ra, rb):
    ga, gb = grid_key(ra), grid_key(rb)
    assert (ga is None) == (gb is None)
    if ga is not None:
        assert torch.equal(ga[0], gb[0]) and torch.equal(ga[1], gb[1])


# ------------------------------------------------------------------------------------------------ 1. the reference run, resumed
def test_driver_loop_resumes_bit_for_bit(pkg, ck, env_golden, loop_golden, tmp_path):
    g, e = loop_golden, env_golden
    maps = (e["speed"], e["angle"])

    def run(loop, record, saves=None):
        upd = []
        real = loop.robot.td3_agent.td3_update

        def update(memory, **kw):
            out = real(memory, **kw)
            upd.append(torch.cat([out[0].reshape(-1), out[1].reshape(-1)]).cpu())
            return out
        loop.robot.td3_agent.td3_update = update
        while not loop.finished:
            if saves is not None:
                for name, due in saves.items():
                    if name not in record["saved"] and due(loop):
                        pkg.save_checkpoint(str(tmp_path / name), loop)
                        record["saved"][name] = (loop.ticks, loop.test_ticks, len(record["kinds"]), len(upd))
            kind = loop.update()
            record["kinds"].append(kind)
            record["states"].append(np.array(loop.state, dtype=np.float64))
            record["money"].append(loop.calculate_remaining_money())
        record["losses"] = upd
        record["final"] = (loop.success, loop.test_ticks, loop.test_best_distance, loop.penalty, loop.ticks, loop.steps_bought,
                           loop.resets_bought, loop.demos_bought, len(loop.robot.memory))
        record["actor"] = loop.robot.td3_agent.actor_network.flat_parameters().cpu().clone()
        record["uniform"] = np.random.uniform()
        return record

    torch.manual_seed(0)
    loop = pkg.DriverLoop.from_seed(1707366464, maps=maps, tick_seconds=float(g["tick_seconds"]))
    saves = {"after_demos": lambda l: l.demos_bought == 3 and l.mode == "training",
             "between_updates": lambda l: l.robot.num_updates == 5 and l.mode == "training",
             "testing": lambda l: l.mode == "testing" and l.test_ticks == 20}
    ref = run(loop, {"kinds": [], "states": [], "money": [], "saved": {}}, saves)
    assert set(ref["saved"]) == set(saves) and ref["final"][0] == bool(g["success"])
    for name, (ticks, test_ticks, at, n_upd) in ref["saved"].items():
        torch.manual_seed(1)
        fresh = pkg.DriverLoop.from_seed(12345, maps=maps, tick_seconds=float(g["tick_seconds"]))   # another seed: other goal, weights, stream
        pkg.load_checkpoint(str(tmp_path / name), fresh)
        assert (fresh.ticks, fresh.test_ticks) == (ticks, test_ticks)
        out = run(fresh, {"kinds": [], "states": [], "money": []})
        assert out["kinds"] == ref["kinds"][at:], name
        assert all(np.array_equal(x, y) for x, y in zip(out["states"], ref["states"][at:])), name
        assert out["money"] == ref["money"][at:], name
        assert len(out["losses"]) == len(ref["losses"]) - n_upd
        for x, y in zip(out["losses"], ref["losses"][n_upd:]):       # losses are summed with atomics: equal up to that rounding
            torch.testing.assert_close(x, y, rtol=1e-6, atol=0)
        assert out["final"] == ref["final"], name
        assert torch.equal(out["actor"], ref["actor"]), name
        assert out["uniform"] == ref["uniform"], name


# ------------------------------------------------------------------------------------------------ 2. BatchedTrainer in every form
FORMS = ["hooks", "fused", "graph8_mt19937", "graph8_philox", "multi_tick", "scheduler_demos", "map_seeds", "maps_bank"]


def make_trainer(pkg, form, n, seed):
    from oracle import env_oracle as eo
    torch.manual_seed(seed)
    speed, angle = eo.synthetic_maps(0)
    kw_env = {"maps": (speed, angle)}
    if form == "map_seeds":
        idx = np.random.RandomState(seed).randint(0, 5, n)
        kw_env = {"map_seeds": [3, 11, 2024, 7, 99], "map_index": idx}
    elif form == "maps_bank":
        s2, a2 = eo.synthetic_maps(1)
        kw_env = {"maps": (np.stack([speed, s2, speed[::-1].copy()]), np.stack([angle, a2, angle.T.copy()]))}
    env = pkg.Environment(num_envs=n, seed=100 + seed, **kw_env)
    robot = pkg.Robot(env._goal.t(), hidden=64, layers=2, seed=seed, buffer_size=1 << 17)
    robot.episodes_per_update = 1 << 30                               # learner off
    if form != "scheduler_demos":
        robot.set_demonstration_states(np.random.RandomState(1).uniform(0, 99, (200, 2)))
    kw = {"hooks": {}, "fused": {"fused": True},
          "graph8_mt19937": {"fused": True, "graph": True, "check_interval": 8},
          "graph8_philox": {"fused": True, "graph": True, "check_interval": 8, "noise": "philox"},
          "multi_tick": {"fused": True, "graph": True, "check_interval": 8, "noise": "philox"},
          "scheduler_demos": {"fused": True, "graph": True, "check_interval": 8, "scheduler": True, "demonstrations": True},
          "map_seeds": {"fused": True, "graph": True, "check_interval": 8},
          "maps_bank": {"fused": True, "graph": True, "check_interval": 8, "noise": "philox"}}[form]
    if form == "multi_tick":
        robot.td3_agent.precision = "f16"
    return pkg.BatchedTrainer(env, robot, **kw)


# a single env plans its demonstrations on the host (Environment.get_demonstration), so the batched demo ticks need n > 1
@pytest.mark.parametrize("form,n", [(f, n) for f in FORMS for n in (1, 4133) if (f, n) != ("scheduler_demos", 1)] + [("scheduler_demos", 2)])
def test_trainer_resumes_bit_for_bit(pkg, form, n, tmp_path):
    K = 24
    tr = make_trainer(pkg, form, n, seed=1)
    tr.run(16)
    path = str(tmp_path / "ckpt.pt")
    pkg.save_checkpoint(path, tr)
    tr.run(K)
    ref = tr.state_dict()
    if form == "multi_tick" and n > 128:
        assert tr._multi_tick_ok()

    fresh = make_trainer(pkg, form, n, seed=2)
    pkg.load_checkpoint(path, fresh)
    fresh.run(K)
    assert_same_state(fresh.state_dict(), ref)
    assert_same_grids(fresh.robot, tr.robot)

    # rollback: the live trainer goes back to the checkpoint and reuses the graphs it has captured
    graphs = (tr._graph, tr._graph_k)
    pkg.load_checkpoint(path, tr)
    tr.run(K)
    assert (tr._graph, tr._graph_k) == graphs
    assert_same_state(tr.state_dict(), ref)


def test_trainer_randn_noise_restores_torch_generator(pkg, tmp_path):
    def make(seed):
        from oracle import env_oracle as eo
        env = pkg.Environment(num_envs=300, seed=5 + seed, maps=eo.synthetic_maps(0))
        robot = pkg.Robot(env._goal.t(), hidden=64, layers=2, seed=seed, buffer_size=1 << 14)
        robot.episodes_per_update = 1 << 30
        return pkg.BatchedTrainer(env, robot, fused=True, noise="randn")
    tr = make(1)
    tr.run(5)
    sd = tr.state_dict()
    tr.run(7)
    ref = tr.state_dict()
    fresh = make(2)
    torch.cuda.manual_seed(999)
    fresh.load_state_dict(sd)
    fresh.run(7)
    assert_same_state(fresh.state_dict(), ref)


def test_async_snapshot_is_folded_into_the_save(pkg, tmp_path):
    """An update decision in flight at the save is taken identically after the load."""
    def make(seed):
        from oracle import env_oracle as eo
        env = pkg.Environment(num_envs=512, seed=5 + seed, maps=eo.synthetic_maps(0))
        robot = pkg.Robot(env._goal.t(), hidden=64, layers=2, seed=seed, buffer_size=1 << 15)
        robot.episodes_per_update = 64
        robot.memory.sampler = "philox"
        agent = robot.td3_agent                                      # updates run but move nothing: the episodes stay the same
        agent.actor_lr = agent.critic_lr = agent.tau = 0.0
        return pkg.BatchedTrainer(env, robot, fused=True, graph=True, check_interval=8, noise="philox", async_check=True)
    tr = make(1)
    tr.run(64)
    assert tr.robot._snap is not None and tr.robot._snap["event"] is not None
    sd = tr.state_dict()
    tr.run(120)
    ref = tr.state_dict()
    assert tr.robot.num_updates > sd["robot"]["host"]["num_updates"]
    fresh = make(2)
    fresh.load_state_dict(sd)
    fresh.run(120)
    out = fresh.state_dict()
    assert out["robot"]["host"]["num_updates"] == ref["robot"]["host"]["num_updates"]
    assert torch.equal(out["robot"]["td3_agent"]["tensors"]["steps"], ref["robot"]["td3_agent"]["tensors"]["steps"])


# ------------------------------------------------------------------------------------------------ 3. the learner
def _filled_replay(pkg, rows, **kw):
    rb = pkg.ReplayBuffer(4096, **kw)
    g = torch.Generator(device="cuda").manual_seed(7)
    s = torch.rand((rows, 2), device="cuda", generator=g) * 98.9999
    a = torch.rand((rows, 2), device="cuda", generator=g) * 10 - 5
    s2 = (s + a).clamp(0, 98.9999)
    r = -torch.linalg.norm(s2 - torch.tensor([80., 20.], device="cuda"), dim=1)
    rb.push(s, a, r, s2, (torch.arange(rows, device="cuda") % 50) == 49)
    return rb


def _agent(pkg, torch_seed, hidden=200, layers=3, precision="fp32"):
    torch.manual_seed(torch_seed)
    td3 = pkg.TD3(pkg.Residual_Actor_Network(hidden, layers), pkg.Residual_Critic_Network(hidden, layers),
                  pkg.Residual_Critic_Network(hidden, layers))
    td3.precision = precision
    return td3


@pytest.mark.parametrize("sampler", ["numpy_global", "seeded", "philox"])
def test_learner_resumes_bit_for_bit(pkg, sampler, tmp_path):
    kw = {} if sampler == "numpy_global" else {"seed": 11}
    np.random.seed(5)
    td3, rb = _agent(pkg, 0), _filled_replay(pkg, 3000, **kw)
    if sampler == "philox":
        rb.sampler = "philox"
    for _ in range(2):
        td3.td3_update(rb)
    pkg.save_checkpoint(str(tmp_path / "td3.pt"), td3)
    pkg.save_checkpoint(str(tmp_path / "rb.pt"), rb)
    l_ref = [x.clone() for x in td3.td3_update(rb)]
    ref = (td3.state_dict(), rb.state_dict(), np.random.get_state()[1].copy())

    fresh, frb = _agent(pkg, 99), _filled_replay(pkg, 10, **kw)
    np.random.seed(77)
    pkg.load_checkpoint(str(tmp_path / "td3.pt"), fresh)
    pkg.load_checkpoint(str(tmp_path / "rb.pt"), frb)
    l_out = fresh.td3_update(frb)
    out = fresh.state_dict()
    out["host"]["last_losses"] = ref[0]["host"]["last_losses"] = None          # compared below, within the atomic sums' rounding
    assert_same_state(out, ref[0])
    assert_same_state(frb.state_dict(), ref[1])
    if sampler == "numpy_global":                                  # the sampler's stream is numpy's: restored by the load
        assert np.array_equal(np.random.get_state()[1], ref[2])
    for a, b in zip(l_out, l_ref):
        torch.testing.assert_close(a, b, rtol=1e-6, atol=0)


@pytest.mark.parametrize("precision", ["f16", "tf32"])
def test_learner_rebuilds_derived_weights(pkg, precision, tmp_path):
    td3, rb = _agent(pkg, 0, 256, 2, precision), _filled_replay(pkg, 3000, seed=3)
    td3.prepare_forward(256)
    td3.td3_update(rb)
    td3.prepare_forward(256)
    sd = td3.state_dict()
    fresh = _agent(pkg, 5, 256, 2, precision)
    fresh.prepare_forward(256)                                      # derived copies of OTHER weights exist: load must rebuild them
    fresh.load_state_dict(sd)
    torch.cuda.synchronize()
    assert torch.equal(fresh.params_t, td3.params_t)
    if precision == "f16":
        assert torch.equal(fresh.params_h, td3.params_h)
    else:
        # [u | v], each one arena long; the optimiser does not keep v of the target networks (they run forward only: nothing reads
        # it), a rebuild writes it - compare everything a kernel reads
        total = td3.params.numel()
        assert torch.equal(fresh.params_u[:total + total // 2], td3.params_u[:total + total // 2])
    x = torch.rand((512, 2), device="cuda") * 50
    assert torch.equal(fresh.forward(0, x), td3.forward(0, x))


# ------------------------------------------------------------------------------------------------ 4. inventory guard
def _tensor_paths(obj, skip):
    from importlib import import_module
    MtBank = import_module("residual-td3-robot-navigation_b200.rng").MtBank

    def walk(v, path):
        if isinstance(v, torch.Tensor):
            yield path
        elif isinstance(v, dict):
            for k, x in v.items():
                yield from walk(x, "%s.%s" % (path, k))
        elif isinstance(v, (list, tuple)):
            for i, x in enumerate(v):
                yield from walk(x, "%s.%d" % (path, i))
        elif isinstance(v, MtBank):
            yield from walk(vars(v), path)
    for name, v in vars(obj).items():
        if not isinstance(v, skip):
            yield from walk(v, name)


def test_every_tensor_is_stored_or_classified(pkg, ck):
    from oracle import env_oracle as eo
    env = pkg.Environment(num_envs=256, seed=3, map_seeds=[1, 2], map_index=np.arange(256) % 2)
    robot = pkg.Robot(env._goal.t(), hidden=64, layers=2, seed=1, buffer_size=1 << 15)
    robot.td3_agent.precision = "f16"
    robot.episodes_per_update = 1 << 30
    tr = pkg.BatchedTrainer(env, robot, fused=True, graph=True, check_interval=4, scheduler=True, demonstrations=True, async_check=True)
    tr.run(12)
    robot.td3_agent.td3_update(robot.memory)
    robot.td3_agent.precision = "tf32"
    robot.td3_agent.prepare_forward(256)
    robot.evaluate(env, max_steps=4)
    robot.td3_agent.precision = "fp32"
    robot.evaluate(env, max_steps=4)
    env.rollout_host(torch.zeros((2, 2, 256)), mode="staged")
    loop = pkg.DriverLoop(pkg.Environment(seed=4, maps=eo.synthetic_maps(0)), pkg.Robot(np.array([80., 20.]), seed=2))
    six = (pkg.ReplayBuffer, pkg.TD3, pkg.Environment, pkg.Robot, pkg.BatchedTrainer, pkg.DriverLoop, pkg.Residual_Actor_Network,
           pkg.Residual_Critic_Network)
    unclassified = []
    for obj in (robot.memory, robot.td3_agent, env, robot, tr, loop):
        cls = type(obj).__name__
        sd = obj.state_dict()
        known = set(sd["tensors"]) | set(sd["host"]) | set(ck.NOT_SAVED[cls])
        for path in _tensor_paths(obj, six):
            parts = path.split(".")
            if not any(".".join(parts[:i]) in known for i in range(1, len(parts) + 1)):
                unclassified.append("%s.%s" % (cls, path))
    assert not unclassified, unclassified


# ------------------------------------------------------------------------------------------------ 5. rejection
def _checksum(tr):
    bits = lambda t: int(t.contiguous().view(-1).view(torch.uint8).to(torch.int64).sum())
    out = [tuple(tr.robot.td3_agent.replica_checksum().tolist())]
    for obj in (tr.env, tr.robot, tr.robot.memory, tr):
        out += [bits(v) for v in vars(obj).values() if isinstance(v, torch.Tensor)]
    out += [bits(v) for k in ("mt", "pos", "has_gauss", "gauss") for v in (getattr(tr.env._bank, k), getattr(tr.robot._bank, k))]
    return out


def test_mismatches_are_rejected_before_anything_is_written(pkg, ck, tmp_path):
    def make(seed, n=256, hidden=64, cap=1 << 14):
        from oracle import env_oracle as eo
        env = pkg.Environment(num_envs=n, seed=seed, maps=eo.synthetic_maps(0))
        robot = pkg.Robot(env._goal.t(), hidden=hidden, layers=2, seed=seed, buffer_size=cap)
        robot.episodes_per_update = 1 << 30
        return pkg.BatchedTrainer(env, robot, fused=True, scheduler=True, demonstrations=True)
    src = make(1)
    src.run(5)
    sd = src.state_dict()
    dst = make(2)
    dst.run(5)
    before = _checksum(dst)
    import copy

    def edited(fn):
        d = copy.deepcopy(sd)
        fn(d)
        return d

    def drop(path):
        def fn(d):
            *head, last = path
            for p in head:
                d = d[p]
            del d[last]
        return fn

    def setv(path, value):
        def fn(d):
            *head, last = path
            for p in head:
                d = d[p]
            d[last] = value(d[last]) if callable(value) else value
        return fn
    bad = {
        "class": edited(setv(("meta", "class"), "DriverLoop")),
        "version": edited(setv(("robot", "td3_agent", "meta", "version"), 999)),
        "world": edited(setv(("robot", "td3_agent", "meta", "world"), 2)),
        "rank": edited(setv(("robot", "td3_agent", "meta", "rank"), 1)),
        "missing key": edited(drop(("robot", "memory", "tensors", "notdone"))),
        "missing bank": edited(drop(("env", "tensors", "_bank.gauss"))),
        "dtype": edited(setv(("robot", "tensors", "_plan_index"), lambda t: t.long())),
        "shape": edited(setv(("robot", "td3_agent", "tensors", "adam_m"), lambda t: t[:-1])),
        "demo count": edited(setv(("robot", "tensors", "_env_demo.count"), lambda t: t + 10 ** 6)),
    }
    for what, d in bad.items():
        with pytest.raises(ValueError):
            dst.load_state_dict(d)
        assert _checksum(dst) == before, what
    for other in (make(3, n=128), make(3, hidden=128), make(3, cap=1 << 15)):    # num_envs, hidden, capacity
        b = _checksum(other)
        with pytest.raises(ValueError):
            other.load_state_dict(sd)
        assert _checksum(other) == b
    with pytest.raises(ValueError):
        dst.env.load_state_dict(sd["robot"])                       # another class
    assert _checksum(dst) == before
    with pytest.raises(TypeError):
        pkg.save_checkpoint(str(tmp_path / "x.pt"), object())

    # an interrupted save leaves the previous file loadable
    path = str(tmp_path / "run.pt")
    pkg.save_checkpoint(path, src)
    src.run(3)
    real = torch.save

    def killed(*a, **k):
        raise RuntimeError("killed part-way")
    torch.save = killed
    try:
        with pytest.raises(RuntimeError):
            pkg.save_checkpoint(path, src)
    finally:
        torch.save = real
    assert os.listdir(tmp_path) == ["run.pt"]
    pkg.load_checkpoint(path, dst)
    assert_same_state(dst.state_dict(), sd)


def test_save_refuses_capture_and_open_sampling_session(pkg):
    rb = _filled_replay(pkg, 500)
    rb.begin_sampling_session()
    try:
        with pytest.raises(RuntimeError, match="session"):
            rb.state_dict()
    finally:
        rb.end_sampling_session()
    td3 = _agent(pkg, 0, 64, 2)
    g = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError, match="capture"):
        with torch.cuda.graph(g):
            td3.state_dict()


# ------------------------------------------------------------------------------------------------ 6. export
class _Net(torch.nn.Module):
    def __init__(self, i, h, layers, o):
        super().__init__()
        dims = [i] + [h] * layers
        for k in range(layers):
            setattr(self, "layer_%d" % (k + 1), torch.nn.Linear(dims[k], dims[k + 1]))
        self.output_layer = torch.nn.Linear(h, o)
        self.layers = layers

    def forward(self, x):
        for k in range(self.layers):
            x = torch.relu(getattr(self, "layer_%d" % (k + 1))(x))
        return self.output_layer(x)


def test_export_networks_load_into_plain_modules(pkg, ck):
    td3, rb = _agent(pkg, 0), _filled_replay(pkg, 3000, seed=4)
    td3.td3_update(rb)
    nets = td3.export_networks()
    assert set(nets) == set(ck.NETWORKS)
    x = torch.rand((300, 4), device="cuda") * 60 - 10
    for k, name in enumerate(ck.NETWORKS):
        i, o = (2, 2) if "actor" in name else (4, 1)
        m = _Net(i, 200, 3, o).double()
        m.load_state_dict({key: v.double() for key, v in nets[name].items()})
        ref = m(x[:, :i].double().cpu())
        got = td3.forward(k, x[:, :i]).double().cpu()
        torch.testing.assert_close(got, ref, rtol=1e-5, atol=1e-5)
    before = td3.params.clone()
    fresh = _agent(pkg, 9)
    fresh.import_networks(nets)
    assert torch.equal(fresh.params, before)
    assert all(torch.equal(a, b) for n in ck.NETWORKS for a, b in zip(fresh.export_networks()[n].values(), nets[n].values()))
    nets["target_actor"]["layer_1.weight"] = nets["target_actor"]["layer_1.weight"][:, :1]
    with pytest.raises(ValueError):
        fresh.import_networks(nets)
    assert torch.equal(fresh.params, before)


# ------------------------------------------------------------------------------------------------ 7. two GPUs
@pytest.mark.parametrize("collective", ["p2p", "nccl"])
def test_data_parallel_checkpoint(collective, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    torchrun = shutil.which("torchrun") or os.path.join(os.path.dirname(sys.executable), "torchrun")
    env = dict(os.environ, RTD3_DP_COLLECTIVE=collective)
    r = subprocess.run([torchrun, "--standalone", "--nproc_per_node=2", os.path.join(ROOT, "tools", "checkpoint_dp_check.py"), str(tmp_path)],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert "checkpoint DP2 OK" in r.stdout
