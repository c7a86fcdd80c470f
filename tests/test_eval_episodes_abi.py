"""rtd3_eval_starts / rtd3_eval_step_episodes / rtd3_eval_run_f16_episodes check their arguments before any launch, and
Robot.evaluate checks `episodes` (no compute calls: runs without a GPU)."""
import ctypes
import types

import pytest
import torch


def _args():
    buf = (ctypes.c_double * 4)()                                 # any non-null address: nothing is launched
    p = ctypes.cast(buf, ctypes.c_void_p)
    return buf, p


def test_eval_starts_rejects_bad_arguments_without_a_gpu(pkg):
    L = pkg._lib.lib()
    buf, p = _args()
    before = pkg._lib.launch_count()

    def call(mt=p, pos=p, region=p, goal=None, E=4, starts=p, base=None, state64=p, n=4):
        bank = pkg._lib.MtBankStruct(mt, pos, p, p, n)
        return L.rtd3_eval_starts(ctypes.byref(bank), region, goal, E, starts, base, state64, None)

    assert L.rtd3_eval_starts(None, p, None, 4, p, None, p, None) == -1 and b"null" in L.rtd3_last_error()
    for kw in ({"mt": None}, {"pos": None}, {"region": None}, {"starts": None}, {"state64": None}):
        assert call(**kw) == -1 and b"null" in L.rtd3_last_error()
    assert call(base=p) == -1 and b"goal" in L.rtd3_last_error()
    for E in (0, -1, 1025):
        assert call(E=E) == -1 and b"E must" in L.rtd3_last_error()
    for E, n in ((2, 1 << 30), (1024, 1 << 21), (1, -1)):
        assert call(E=E, n=n) == -1 and b"E * n" in L.rtd3_last_error()
    assert call(n=0) == 0                                           # nothing to draw
    assert pkg._lib.launch_count() == before


def test_eval_step_episodes_rejects_bad_arguments_without_a_gpu(pkg):
    L = pkg._lib.lib()
    buf, p = _args()
    before = pkg._lib.launch_count()

    def call(h=None, goal=p, E=3, xs=p, res=p, base=p, succ=p, steps=p, best=p, traj=None, record=0, n=4, T=10):
        return L.rtd3_eval_step_episodes(h, goal, E, xs, res, base, succ, steps, best, traj, record, n, T, None)

    for kw in ({"goal": None}, {"xs": None}, {"succ": None}, {"steps": None}, {"best": None}):
        assert call(**kw) == -1 and b"null" in L.rtd3_last_error()
    for kw in ({"res": None}, {"base": None}):
        assert call(**kw) == -1 and b"residual" in L.rtd3_last_error()
    assert call(n=-1) == -1 and b"n must" in L.rtd3_last_error()
    for T in (0, -3, 1 << 30):
        assert call(T=T) == -1 and b"T must" in L.rtd3_last_error()
    assert call(traj=p, record=0) == -1 and b"record" in L.rtd3_last_error()
    assert call(traj=None, record=1) == -1 and b"record" in L.rtd3_last_error()
    for E in (0, -1, 1025):
        assert call(E=E) == -1 and b"E must" in L.rtd3_last_error()
    for E, n in ((2, 1 << 30), (1024, 1 << 21)):
        assert call(E=E, n=n) == -1 and b"E * n" in L.rtd3_last_error()
    assert call() == -1 and b"dynamics map" in L.rtd3_last_error()        # no environment handle
    assert call(n=0) == -1                                                  # checked even when there is nothing to do
    assert pkg._lib.launch_count() == before


def test_eval_run_f16_episodes_rejects_bad_arguments_without_a_gpu(pkg):
    L = pkg._lib.lib()
    buf, p = _args()
    before = pkg._lib.launch_count()

    def call(h=None, hidden=128, layers=2, params=p, params_h=p, goal=p, starts=p, E=3, x=p, y=p, succ=p, steps=p, best=p, traj=None,
             record=0, n=4, T=10, work=p):
        return L.rtd3_eval_run_f16_episodes(h, hidden, layers, params, params_h, goal, starts, E, x, y, succ, steps, best, traj, record, n, T,
                                            work, None)

    for kw in ({"goal": None}, {"x": None}, {"y": None}, {"succ": None}, {"steps": None}, {"best": None}):
        assert call(**kw) == -1 and b"null" in L.rtd3_last_error()
    assert call(starts=None) == -1 and b"start planes" in L.rtd3_last_error()
    for kw in ({"params": None}, {"params_h": None}, {"work": None}):
        assert call(**kw) == -1 and b"null parameters" in L.rtd3_last_error()
    assert call(n=-1) == -1 and b"n must" in L.rtd3_last_error()
    for T in (0, 1 << 30):
        assert call(T=T) == -1 and b"T must" in L.rtd3_last_error()
    assert call(traj=p, record=0) == -1 and b"record" in L.rtd3_last_error()
    assert call(traj=None, record=1) == -1 and b"record" in L.rtd3_last_error()
    for E in (0, -1, 1025):
        assert call(E=E) == -1 and b"E must" in L.rtd3_last_error()
    for E, n in ((2, 1 << 30), (1024, 1 << 21)):
        assert call(E=E, n=n) == -1 and b"E * n" in L.rtd3_last_error()
    for hidden, layers in ((200, 2), (32, 2), (288, 2), (128, 3)):
        assert call(hidden=hidden, layers=layers) == -1 and b"layers == 2" in L.rtd3_last_error()
    assert call() == -1 and b"dynamics map" in L.rtd3_last_error()
    assert pkg._lib.launch_count() == before


def test_evaluate_rejects_bad_episodes_without_a_gpu(pkg):
    """The checks run before anything touches the device: a stand-in Robot and environment are enough."""
    robot = types.SimpleNamespace(device=torch.device("cpu"))
    env = types.SimpleNamespace(device=torch.device("cpu"), num_envs=8)
    for bad in (0, -1, 1025, 1.0, 2.5, True, "4", [4]):
        with pytest.raises(ValueError, match="episodes"):
            pkg.Robot.evaluate(robot, env, episodes=bad)
    big = types.SimpleNamespace(device=torch.device("cpu"), num_envs=1 << 21)
    with pytest.raises(ValueError, match="below 2"):
        pkg.Robot.evaluate(robot, big, episodes=1024)
    with pytest.raises(ValueError, match="max_steps"):
        pkg.Robot.evaluate(robot, env, max_steps=0, episodes=4)
