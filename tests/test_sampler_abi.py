"""rtd3_sample_indices_mt19937 / rtd3_sample_indices_philox check their arguments before any launch, and count = 0 draws
nothing (no compute calls: runs without a GPU)."""
import ctypes


def _args():
    buf = (ctypes.c_double * 4)()                                 # any non-null address: nothing is launched
    p = ctypes.cast(buf, ctypes.c_void_p)
    return buf, p


def test_sample_indices_mt19937_rejects_bad_arguments_without_a_gpu(pkg):
    L = pkg._lib.lib()
    buf, p = _args()
    before = pkg._lib.launch_count()

    def call(mt=p, pos=p, streams=5, stream_id=0, n=100, batch=10, count=3, out=p, scratch=p):
        bank = pkg._lib.MtBankStruct(mt, pos, p, p, streams)
        return L.rtd3_sample_indices_mt19937(ctypes.byref(bank), stream_id, n, batch, count, out, scratch, None)

    def err():
        return L.rtd3_last_error()

    assert L.rtd3_sample_indices_mt19937(None, 0, 100, 10, 3, p, p, None) == -1 and b"null" in err()
    for kw in ({"mt": None}, {"pos": None}, {"out": None}):
        assert call(**kw) == -1 and b"null" in err()
    for sid in (-1, 5, 1 << 40):                                    # [0, bank.n) of a bank of five streams
        assert call(stream_id=sid) == -1 and b"stream id" in err()
    assert call(streams=0) == -1 and b"stream id" in err()
    for n, batch in ((100, 0), (100, -1), (100, 101), (1, 2), (0, 1), (-5, 1)):
        assert call(n=n, batch=batch) == -1 and b"batch <= n" in err()
    assert call(count=-1) == -1 and b"batch <= n" in err()
    for n in (56001, 1 << 20, (1 << 31) - 1):
        assert call(n=n) == -1 and b"56000" in err()
    # count * n < 2^30 raw draws: 56 000 * 19 173 < 2^30 <= 56 000 * 19 174 (the first passes and stops at the null scratch)
    assert call(n=56000, count=19174) == -1 and b"2^30" in err()
    assert call(n=1 << 14, count=1 << 16) == -1 and b"2^30" in err()
    assert call(n=56000, count=19173, scratch=None) == -1 and b"scratch" in err()
    for count in (1, 150):
        assert call(count=count, scratch=None) == -1 and b"scratch" in err()
    # count = 0 draws nothing: no launch, no scratch needed, whatever n and the batch are within their limits
    assert call(count=0, scratch=None) == 0
    assert call(n=56000, batch=56000, count=0, scratch=None) == 0
    assert call(n=1, batch=1, count=0, stream_id=4) == 0
    assert pkg._lib.launch_count() == before


def test_sample_indices_philox_rejects_bad_arguments_without_a_gpu(pkg):
    """Philox draws with replacement, so it takes any n in [1, 2^31) and a batch larger than n; there is no bank and no
    scratch.  What it cannot take is rejected before the launch."""
    L = pkg._lib.lib()
    buf, p = _args()
    before = pkg._lib.launch_count()

    def call(seed=0x5eed, offset=0, n=100, batch=10, count=3, out=p):
        return L.rtd3_sample_indices_philox(seed, offset, n, batch, count, out, None)

    assert call(out=None) == -1 and b"bad argument" in L.rtd3_last_error()
    for n in (0, -1, 1 << 31, 1 << 40):
        assert call(n=n) == -1 and b"bad argument" in L.rtd3_last_error()
    for batch in (0, -1):
        assert call(batch=batch) == -1 and b"bad argument" in L.rtd3_last_error()
    assert call(count=-1) == -1 and b"bad argument" in L.rtd3_last_error()
    assert call(count=0) == 0                                       # nothing to draw
    assert call(n=(1 << 31) - 1, batch=1 << 20, count=0, seed=(1 << 64) - 1, offset=(1 << 64) - 1) == 0
    assert pkg._lib.launch_count() == before
