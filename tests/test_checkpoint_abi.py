"""rtd3_robot_demo_grids checks its arguments before any launch, and checkpoint files are rejected before anything is loaded (no
compute calls: runs without a GPU)."""
import ctypes

import pytest


def test_demo_grids_rejects_bad_arguments_without_a_gpu(pkg):
    L = pkg._lib.lib()
    buf = (ctypes.c_double * 4)()                                 # any non-null address: nothing is launched
    p = ctypes.cast(buf, ctypes.c_void_p)
    before = pkg._lib.launch_count()

    def call(sets=p, count=p, cap=8, n=4, sorted_=p, cells=p):
        return L.rtd3_robot_demo_grids(sets, count, cap, n, sorted_, cells, None)

    for kw in ({"sets": None}, {"count": None}, {"sorted_": None}, {"cells": None}):
        assert call(**kw) == -1 and b"null" in L.rtd3_last_error()
    for cap in (0, -1):
        assert call(cap=cap) == -1 and b"cap must" in L.rtd3_last_error()
    for n in (-1, 1 << 31):
        assert call(n=n) == -1 and b"n must" in L.rtd3_last_error()
    assert call(n=0) == 0                                         # nothing to do
    assert call(sets=None, n=0) == -1                             # checked even when there is nothing to do
    with pytest.raises(pkg._lib.Rtd3Error):
        pkg._lib.check(call(cap=0), "robot_demo_grids")
    assert pkg._lib.launch_count() == before


def test_demo_grids_is_bound_like_the_header(pkg):
    assert "rtd3_robot_demo_grids" in pkg._lib.exported_symbols()


def test_checkpoint_files_of_another_kind_are_rejected(pkg, tmp_path):
    import torch
    from importlib import import_module
    ck = import_module("residual-td3-robot-navigation_b200.checkpoint")
    bad = tmp_path / "other.pt"
    torch.save({"meta": {"format": "something else"}, "state": {}}, bad)
    with pytest.raises(ValueError):
        ck._read(str(bad))
    old = tmp_path / "old.pt"
    torch.save({"meta": {"format": ck.FORMAT, "version": ck.FORMAT_VERSION + 1}, "state": {}}, old)
    with pytest.raises(ValueError, match="version"):
        ck._read(str(old))


def test_atomic_save_keeps_the_old_file_when_interrupted(pkg, tmp_path, monkeypatch):
    import torch
    from importlib import import_module
    ck = import_module("residual-td3-robot-navigation_b200.checkpoint")
    path = tmp_path / "ckpt.pt"
    ck._atomic_save({"meta": {"format": ck.FORMAT, "version": ck.FORMAT_VERSION}, "state": {"x": torch.arange(3)}}, str(path))

    def killed(*a, **k):
        raise KeyboardInterrupt("killed part-way")
    monkeypatch.setattr(torch, "save", killed)
    with pytest.raises(KeyboardInterrupt):
        ck._atomic_save({"meta": {}, "state": {"x": torch.arange(5)}}, str(path))
    monkeypatch.undo()
    assert sorted(p.name for p in tmp_path.iterdir()) == ["ckpt.pt"]          # no temporary file left behind
    assert torch.equal(ck._read(str(path))["state"]["x"], torch.arange(3))
