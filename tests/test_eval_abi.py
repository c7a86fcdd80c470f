"""rtd3_eval_step / rtd3_eval_run_f16 check their arguments before any launch (no compute calls: runs without a GPU)."""
import ctypes

import pytest


def _args():
    buf = (ctypes.c_double * 4)()                                 # any non-null address: nothing is launched
    p = ctypes.cast(buf, ctypes.c_void_p)
    return buf, p


def test_eval_step_rejects_bad_arguments_without_a_gpu(pkg):
    L = pkg._lib.lib()
    buf, p = _args()
    before = pkg._lib.launch_count()

    def call(h=None, goal=p, x=p, y=p, res=p, base=p, succ=p, steps=p, best=p, traj=None, record=0, n=4, T=10):
        return L.rtd3_eval_step(h, goal, x, y, res, base, succ, steps, best, traj, record, n, T, None)

    for kw in ({"goal": None}, {"x": None}, {"y": None}, {"succ": None}, {"steps": None}, {"best": None}):
        assert call(**kw) == -1
        assert b"null" in L.rtd3_last_error()
    for kw in ({"res": None}, {"base": None}):
        assert call(**kw) == -1
        assert b"residual" in L.rtd3_last_error()
    assert call(n=-1) == -1 and b"n must" in L.rtd3_last_error()
    assert call(n=1 << 31) == -1 and b"n must" in L.rtd3_last_error()
    for T in (0, -3, 1 << 30):
        assert call(T=T) == -1 and b"T must" in L.rtd3_last_error()
    assert call(traj=p, record=0) == -1 and b"record" in L.rtd3_last_error()
    assert call(traj=None, record=1) == -1 and b"record" in L.rtd3_last_error()
    assert call() == -1 and b"dynamics map" in L.rtd3_last_error()        # no environment handle
    assert call(n=0) == -1                                                  # checked even when there is nothing to do
    with pytest.raises(pkg._lib.Rtd3Error):
        pkg._lib.check(call(T=0), "eval_step")
    assert pkg._lib.launch_count() == before


def test_eval_run_f16_rejects_bad_arguments_without_a_gpu(pkg):
    L = pkg._lib.lib()
    buf, p = _args()
    before = pkg._lib.launch_count()

    def call(h=None, hidden=128, layers=2, params=p, params_h=p, goal=p, x=p, y=p, succ=p, steps=p, best=p, traj=None, record=0, n=4,
             T=10, work=p):
        return L.rtd3_eval_run_f16(h, hidden, layers, params, params_h, goal, x, y, succ, steps, best, traj, record, n, T, work, None)

    for kw in ({"goal": None}, {"x": None}, {"y": None}, {"succ": None}, {"steps": None}, {"best": None}):
        assert call(**kw) == -1
        assert b"null" in L.rtd3_last_error()
    for kw in ({"params": None}, {"params_h": None}, {"work": None}):
        assert call(**kw) == -1
        assert b"null parameters" in L.rtd3_last_error()
    assert call(n=-1) == -1 and b"n must" in L.rtd3_last_error()
    for T in (0, 1 << 30):
        assert call(T=T) == -1 and b"T must" in L.rtd3_last_error()
    assert call(traj=p, record=0) == -1 and b"record" in L.rtd3_last_error()
    assert call(traj=None, record=1) == -1 and b"record" in L.rtd3_last_error()
    for hidden, layers in ((200, 2), (32, 2), (288, 2), (128, 3), (128, 1)):
        assert call(hidden=hidden, layers=layers) == -1
        assert b"layers == 2" in L.rtd3_last_error()
    assert call() == -1 and b"dynamics map" in L.rtd3_last_error()
    assert pkg._lib.launch_count() == before
