"""rtd3_perlin_maps checks its arguments before any launch (no compute calls: runs without a GPU)."""
import ctypes

import pytest


def test_perlin_maps_rejects_bad_arguments_without_a_gpu(pkg):
    L = pkg._lib.lib()
    buf = (ctypes.c_double * 4)()                                 # any non-null address: nothing is launched
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert L.rtd3_perlin_maps(None, 1, p, p, None) == -1
    assert b"null" in L.rtd3_last_error()
    assert L.rtd3_perlin_maps(p, 1, None, p, None) == -1
    assert L.rtd3_perlin_maps(p, 1, p, None, None) == -1
    for K in (0, -1, 65537):
        assert L.rtd3_perlin_maps(p, K, p, p, None) == -1
        assert b"65536" in L.rtd3_last_error()
    with pytest.raises(pkg._lib.Rtd3Error):
        pkg._lib.check(L.rtd3_perlin_maps(p, 0, p, p, None), "perlin_maps")


def test_map_seeds_with_maps_is_rejected_before_any_device_work(pkg):
    speed, angle = pkg.synthetic_maps(0)
    with pytest.raises(ValueError):
        pkg.Environment(num_envs=4, maps=(speed, angle), map_seeds=[1, 2])


@pytest.mark.parametrize("bad", [[-1], [1, -5], [1.0, 2.0], [[1, 2]], [], [2 ** 63], [2 ** 64], [True, False]])
def test_seed_checks_without_a_gpu(pkg, bad):
    """The seed checks run on the host, before any device work."""
    with pytest.raises(ValueError):
        pkg.environment._checked_seeds(bad)


def test_seed_inputs_without_a_gpu(pkg):
    import numpy as np
    import torch
    check = pkg.environment._checked_seeds
    for bad in (torch.tensor([-1]), torch.tensor([1.0]), torch.tensor([[1]]), torch.zeros(0, dtype=torch.int64), torch.tensor([True]),
                np.zeros(65537, np.int64), np.array([2 ** 63], np.uint64)):
        with pytest.raises(ValueError):
            check(bad)
    assert check(np.array([0, 2 ** 63 - 1], np.uint64)).tolist() == [0, 2 ** 63 - 1]
    assert check(torch.tensor([3, 1], dtype=torch.int32)).dtype == torch.int64
    t = torch.tensor([5])
    check(t)[0] = 7                                               # the checked seeds are a copy
    assert int(t[0]) == 5
