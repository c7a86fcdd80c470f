"""Background checkpoints on the B200: `save_checkpoint(path, obj, background=True)` snapshots the stored state in device memory and
returns; a writer thread copies it to the host and writes the file while the run goes on.  The file must hold the state at the
call, bit for bit (replay rows as multisets, as in test_checkpoint_gpu.py), and the run must continue exactly as without the save."""
import os
import shutil
import subprocess
import sys
import threading
from importlib import import_module

import numpy as np
import pytest
import torch

from test_checkpoint_gpu import FORMS, assert_same_state, make_trainer

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ck():
    return import_module("residual-td3-robot-navigation_b200.checkpoint")


def _differs(a, b):
    """Whether two state dicts differ anywhere (so a snapshot taken late would be caught)."""
    try:
        assert_same_state(a, b)
    except AssertionError:
        return True
    return False


def _advance(tr):
    """Ticks and one learner update after the save: the run's state moves on (in scheduler_demos, a demonstration comes first)."""
    tr.run(24 + 128 // tr.n)                      # at least one batch of replay rows for the update
    if len(tr.robot.memory) > 56000:              # the exact sampler's limit; the sampler mode is stored, so it changes too
        tr.robot.memory.sampler = "philox"
    tr.robot.td3_agent.td3_update(tr.robot.memory)


# ------------------------------------------------------------------------------------------------ 1. the file is the state at the call
@pytest.mark.parametrize("form,n", [(f, n) for f in FORMS for n in (1, 4133) if (f, n) != ("scheduler_demos", 1)] + [("scheduler_demos", 2)])
def test_background_file_is_the_state_at_the_call(pkg, ck, form, n, tmp_path):
    tr = make_trainer(pkg, form, n, seed=1)
    tr.run(1 if form == "scheduler_demos" else 16)   # the scheduler's demonstrations are the first three ticks
    sd = tr.state_dict()
    path = str(tmp_path / "bg.pt")
    p = pkg.save_checkpoint(path, tr, background=True)
    assert isinstance(p, pkg.PendingCheckpoint) and p.path == path
    _advance(tr)
    if form == "scheduler_demos":
        assert int(tr.demos_bought.sum()) > int(sd["tensors"]["demos_bought"].sum())
    assert p.wait() == path and p.done()
    assert _differs(tr.state_dict(), sd)
    assert_same_state(ck._read(path)["state"], sd)
    fresh = make_trainer(pkg, form, n, seed=2)
    pkg.load_checkpoint(path, fresh)
    assert_same_state(fresh.state_dict(), sd)


def _filled_replay(pkg, rows, **kw):
    rb = pkg.ReplayBuffer(4096, **kw)
    g = torch.Generator(device="cuda").manual_seed(7)
    s = torch.rand((rows, 2), device="cuda", generator=g) * 98.9999
    a = torch.rand((rows, 2), device="cuda", generator=g) * 10 - 5
    s2 = (s + a).clamp(0, 98.9999)
    r = -torch.linalg.norm(s2 - torch.tensor([80., 20.], device="cuda"), dim=1)
    rb.push(s, a, r, s2, (torch.arange(rows, device="cuda") % 50) == 49)
    return rb


def _agent(pkg, torch_seed, hidden=200, layers=3):
    torch.manual_seed(torch_seed)
    return pkg.TD3(pkg.Residual_Actor_Network(hidden, layers), pkg.Residual_Critic_Network(hidden, layers),
                   pkg.Residual_Critic_Network(hidden, layers))


@pytest.mark.parametrize("sampler", ["numpy_global", "seeded", "philox"])
def test_background_learner_file_is_the_state_at_the_call(pkg, ck, sampler, tmp_path):
    kw = {} if sampler == "numpy_global" else {"seed": 11}
    np.random.seed(5)
    td3, rb = _agent(pkg, 0), _filled_replay(pkg, 3000, **kw)
    if sampler == "philox":
        rb.sampler = "philox"
    td3.td3_update(rb)
    sd = (td3.state_dict(), rb.state_dict())
    p_td3 = pkg.save_checkpoint(str(tmp_path / "td3.pt"), td3, background=True)
    p_rb = pkg.save_checkpoint(str(tmp_path / "rb.pt"), rb, background=True)
    for _ in range(2):                                             # weights, moments, clocks, losses and the sampler's stream move on
        td3.td3_update(rb)
    p_td3.wait()
    p_rb.wait()
    assert _differs(td3.state_dict(), sd[0]) and _differs(rb.state_dict(), sd[1])
    assert_same_state(ck._read(p_td3.path)["state"], sd[0])
    assert_same_state(ck._read(p_rb.path)["state"], sd[1])
    fresh, frb = _agent(pkg, 99), _filled_replay(pkg, 10, **kw)
    pkg.load_checkpoint(p_td3.path, fresh)
    pkg.load_checkpoint(p_rb.path, frb)
    assert_same_state(fresh.state_dict(), sd[0])
    assert_same_state(frb.state_dict(), sd[1])


# ------------------------------------------------------------------------------------------------ 2. the reference run is not perturbed
def _drive(pkg, loop, record, saves=None, tmp_path=None):
    """The reference run through DriverLoop (as test_checkpoint_gpu.py's resume test), with background saves where `saves` says."""
    upd = []
    real = loop.robot.td3_agent.td3_update

    def update(memory, **kw):
        out = real(memory, **kw)
        upd.append(torch.cat([out[0].reshape(-1), out[1].reshape(-1)]).cpu())
        return out
    loop.robot.td3_agent.td3_update = update
    pending = []
    while not loop.finished:
        if saves is not None:
            for name, due in saves.items():
                if name not in record["saved"] and due(loop):
                    pending.append(pkg.save_checkpoint(str(tmp_path / name), loop, background=True))
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
    for p in pending:
        p.wait()
    return record


def _same_run(out, ref, at=0, n_upd=0, what=""):
    assert out["kinds"] == ref["kinds"][at:], what
    assert all(np.array_equal(x, y) for x, y in zip(out["states"], ref["states"][at:])), what
    assert len(out["states"]) == len(ref["states"]) - at, what
    assert out["money"] == ref["money"][at:], what
    assert len(out["losses"]) == len(ref["losses"]) - n_upd, what
    for x, y in zip(out["losses"], ref["losses"][n_upd:]):      # losses are summed with atomics: equal up to that rounding
        torch.testing.assert_close(x, y, rtol=1e-6, atol=0)
    assert out["final"] == ref["final"], what
    assert torch.equal(out["actor"], ref["actor"]), what
    assert out["uniform"] == ref["uniform"], what


def test_background_saves_leave_the_reference_run_unchanged(pkg, env_golden, loop_golden, tmp_path):
    g, e = loop_golden, env_golden
    maps = (e["speed"], e["angle"])

    def make(seed, torch_seed):
        torch.manual_seed(torch_seed)
        return pkg.DriverLoop.from_seed(seed, maps=maps, tick_seconds=float(g["tick_seconds"]))
    plain = _drive(pkg, make(1707366464, 0), {"kinds": [], "states": [], "money": []})
    saves = {"after_demos": lambda l: l.demos_bought == 3 and l.mode == "training",
             "between_updates": lambda l: l.robot.num_updates == 5 and l.mode == "training",
             "testing": lambda l: l.mode == "testing" and l.test_ticks == 20}
    ref = _drive(pkg, make(1707366464, 0), {"kinds": [], "states": [], "money": [], "saved": {}}, saves, tmp_path)
    assert set(ref["saved"]) == set(saves) and ref["final"][0] == bool(g["success"])
    _same_run(ref, plain, what="with background saves")
    for name, (ticks, test_ticks, at, n_upd) in ref["saved"].items():
        fresh = make(12345, 1)                                     # another seed: other goal, weights, stream
        pkg.load_checkpoint(str(tmp_path / name), fresh)
        assert (fresh.ticks, fresh.test_ticks) == (ticks, test_ticks)
        _same_run(_drive(pkg, fresh, {"kinds": [], "states": [], "money": []}), ref, at, n_upd, name)


# ------------------------------------------------------------------------------------------------ 3. the call returns before the write
def test_the_call_returns_before_the_file_is_written(pkg, ck, tmp_path, monkeypatch):
    tr = make_trainer(pkg, "graph8_philox", 4133, seed=1)
    tr.run(16)
    sd = tr.state_dict()
    entered, release = threading.Event(), threading.Event()
    real = ck._atomic_save

    def blocked(payload, path):
        entered.set()
        if not release.wait(600):
            raise TimeoutError("not released")
        real(payload, path)
    monkeypatch.setattr(ck, "_atomic_save", blocked)
    path = str(tmp_path / "bg.pt")
    p = pkg.save_checkpoint(path, tr, background=True)
    try:
        assert entered.wait(600)                                   # the writer holds the snapshot on the host and waits to write
        ticks = tr.ticks
        tr.run(24)
        torch.cuda.current_stream().synchronize()
        assert tr.ticks == ticks + 24
        assert not p.done() and not os.path.exists(path)
    finally:
        release.set()
    assert p.wait() == path and p.done()
    assert_same_state(ck._read(path)["state"], sd)


# ------------------------------------------------------------------------------------------------ 4. failures
def test_a_failed_write_keeps_the_previous_file_and_frees_the_staging(pkg, ck, tmp_path, monkeypatch):
    tr = make_trainer(pkg, "fused", 4133, seed=1)
    tr.run(16)
    path = str(tmp_path / "run.pt")
    pkg.save_checkpoint(path, tr)
    old = ck._read(path)["state"]
    tr.run(8)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()

    def killed(*a, **k):
        raise RuntimeError("killed part-way")
    monkeypatch.setattr(torch, "save", killed)
    p = pkg.save_checkpoint(path, tr, background=True)
    with pytest.raises(RuntimeError, match="killed part-way"):
        p.wait()
    monkeypatch.undo()
    assert p.done()
    with pytest.raises(RuntimeError, match="killed part-way"):     # kept: every wait() reports it
        p.wait()
    assert torch.cuda.memory_allocated() == before
    assert os.listdir(tmp_path) == ["run.pt"]
    fresh = make_trainer(pkg, "fused", 4133, seed=2)
    pkg.load_checkpoint(path, fresh)
    assert_same_state(fresh.state_dict(), old)


def test_too_little_device_memory_refuses_before_anything_is_done(pkg, ck, tmp_path, monkeypatch):
    tr = make_trainer(pkg, "fused", 4133, seed=1)
    tr.run(8)
    torch.cuda.synchronize()
    before, threads = torch.cuda.memory_allocated(), threading.active_count()
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (1 << 20, 1 << 40))
    path = str(tmp_path / "bg.pt")
    with pytest.raises(RuntimeError, match="device memory"):
        pkg.save_checkpoint(path, tr, background=True)
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == before and threading.active_count() == threads
    assert os.listdir(tmp_path) == []
    monkeypatch.undo()
    pkg.save_checkpoint(path, tr, background=True).wait()          # with the memory there, the same call saves


def test_background_save_refuses_capture_and_open_sampling_session(pkg, tmp_path):
    rb = _filled_replay(pkg, 500)
    rb.begin_sampling_session()
    try:
        with pytest.raises(RuntimeError, match="session"):
            pkg.save_checkpoint(str(tmp_path / "rb.pt"), rb, background=True)
    finally:
        rb.end_sampling_session()
    td3 = _agent(pkg, 0, 64, 2)
    g = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError, match="capture"):
        with torch.cuda.graph(g):
            pkg.save_checkpoint(str(tmp_path / "td3.pt"), td3, background=True)
    assert os.listdir(tmp_path) == []


def test_back_to_back_background_saves(pkg, ck, tmp_path):
    tr = make_trainer(pkg, "graph8_mt19937", 4133, seed=1)
    tr.run(16)
    sd1 = tr.state_dict()
    p1 = pkg.save_checkpoint(str(tmp_path / "a.pt"), tr, background=True)
    tr.run(8)
    sd2 = tr.state_dict()
    p2 = pkg.save_checkpoint(str(tmp_path / "b.pt"), tr, background=True)
    assert p1.done()                                               # the second save waited for the first writer
    tr.run(8)
    assert p2.wait() and p1.wait()
    assert _differs(sd1, sd2)
    assert_same_state(ck._read(p1.path)["state"], sd1)
    assert_same_state(ck._read(p2.path)["state"], sd2)


# ------------------------------------------------------------------------------------------------ 5. exit with a save pending
EXIT_SCRIPT = r"""
import sys, time
sys.path[:0] = [%(root)r, %(tests)r]
import torch
import rtd3_b200 as rt
from importlib import import_module
from test_checkpoint_gpu import make_trainer
ck = import_module("residual-td3-robot-navigation_b200.checkpoint")
tr = make_trainer(rt, "fused", 4133, 1)
tr.run(16)
torch.save(tr.state_dict(), %(ref)r)
real = ck._atomic_save
def slow(payload, path):
    time.sleep(3.0)
    real(payload, path)
ck._atomic_save = slow
p = rt.save_checkpoint(%(path)r, tr, background=True)
tr.run(8)
print("pending at exit:", not p.done(), flush=True)
"""


def test_exit_with_a_pending_save_finishes_the_file(ck, tmp_path):
    path, ref = str(tmp_path / "bg.pt"), str(tmp_path / "ref.pt")
    script = EXIT_SCRIPT % {"root": ROOT, "tests": os.path.join(ROOT, "tests"), "path": path, "ref": ref}
    r = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert "pending at exit: True" in r.stdout
    assert_same_state(ck._read(path)["state"], torch.load(ref, weights_only=True))
    assert sorted(os.listdir(tmp_path)) == ["bg.pt", "ref.pt"]


# ------------------------------------------------------------------------------------------------ 6. two GPUs
@pytest.mark.parametrize("collective", ["p2p", "nccl"])
def test_data_parallel_background_checkpoint(collective, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    torchrun = shutil.which("torchrun") or os.path.join(os.path.dirname(sys.executable), "torchrun")
    env = dict(os.environ, RTD3_DP_COLLECTIVE=collective)
    r = subprocess.run([torchrun, "--standalone", "--nproc_per_node=2", os.path.join(ROOT, "tools", "checkpoint_bg_dp_check.py"),
                        str(tmp_path)], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert "checkpoint background DP2 OK" in r.stdout
