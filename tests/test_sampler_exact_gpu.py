"""The replay index samplers of csrc/rtd3_sample.cu against exact references, at every limit they accept.

Exact sampler (`rtd3_sample_indices_mt19937`, `ReplayBuffer.sample_indices`): numpy's own `RandomState`.  After every device
call the indices `[count, B]` equal `count` calls of `choice(n, B, replace=False)`, AND the bank's 624 key words and position
equal `get_state()`: the kernel writes the stream back as an untempered block plus numpy's position convention, and a stream
that ends on the last word of a block takes its own branch there (position 624 in the block before).  Covered: n up to the
56 000-row limit, full permutations, the 150 draws of an update, start positions 0, 1, 623, 624, samples that end on the last
and on the first word of a block, a multi-stream bank through the C ABI and numpy's global stream (cached Gaussian included).

Philox sampler (`rtd3_sample_indices_philox`, `ReplayBuffer.sampler = "philox"`): out[4t + k] = (r_k * n) >> 32 with
r = Philox4x32-10((c lo, c hi, 0, 0), (seed lo, seed hi)), c = offset + t, restated on uint64 and pinned to oracle/philox.py;
the host advances the offset by ceil(count * B / 4) per call.
"""
import math

import numpy as np
import pytest
import torch

from oracle import philox

pytestmark = pytest.mark.gpu
MT_N = 624
MAX_N = 56000                                       # the exact sampler's limit: the trace kernel keeps n int32 in shared memory


# ------------------------------------------------------------------------------------------------ exact sampler: helpers
def random_key(seed):
    """624 arbitrary key words (any key is a valid numpy state)."""
    return np.random.RandomState(seed).randint(0, 1 << 32, MT_N, dtype=np.uint64).astype(np.uint32)


def numpy_at(key, pos, has_gauss=0, gauss=0.0):
    rs = np.random.RandomState(0)
    rs.set_state(("MT19937", np.asarray(key, np.uint32), int(pos), int(has_gauss), float(gauss)))
    return rs


def replay(pkg, n, seed=1):
    """A seeded replay buffer holding exactly n rows (its draws come from its own bank, not numpy's global stream)."""
    rb = pkg.ReplayBuffer(max(n, 1), seed=seed)
    if n:
        z = torch.zeros((n, 2), dtype=torch.float32, device="cuda")
        rb.push(z, z, z[:, 0], z, torch.zeros(n, dtype=torch.bool, device="cuda"))
    assert len(rb) == n
    return rb


def put_state(rb, key, pos):
    """The stream (key, pos) in a RandomState and in the replay buffer's bank, written as MtBank.sync_from_numpy writes it."""
    rb._bank.mt[:, 0] = torch.from_numpy(np.asarray(key, np.uint32).view(np.int32)).cuda()
    rb._bank.pos[0] = int(pos)
    return numpy_at(key, pos)


def assert_stream(bank, stream, rs):
    _, key, pos, _, _ = rs.get_state()
    got = bank.mt[:, stream].cpu().numpy().view(np.uint32)
    bad = np.nonzero(got != key)[0]
    assert bad.size == 0, "key words %s... differ from numpy's (%d of 624)" % (bad[:6].tolist(), bad.size)
    assert int(bank.pos[stream]) == pos, "position %d, numpy's %d" % (int(bank.pos[stream]), pos)


def draw(rb, rs, B, count):
    """One device call against `count` numpy draws: indices and the whole stream afterwards.  Returns numpy's position."""
    n = len(rb)
    got = rb.sample_indices(B, count).cpu().numpy()
    exp = np.stack([rs.choice(n, B, replace=False) for _ in range(count)])
    assert got.shape == exp.shape
    bad = np.argwhere(got != exp)
    assert bad.size == 0, "n=%d B=%d count=%d: %d indices differ, first at [sample, slot] %s" % (n, B, count, len(bad), bad[0].tolist())
    assert_stream(rb._bank, 0, rs)
    return rs.get_state()[2]


# (n, count, end position, after) -> (key seed, start position): what find_start's search found from (1, 0)
START_HINTS = {(2, 1, 624, None): (1, 623), (3, 1, 624, None): (1, 622), (100, 3, 624, None): (4, 199), (4097, 1, 624, None): (2, 533),
               (10000, 2, 624, None): (20, 79), (32769, 1, 624, None): (69, 9), (56000, 1, 624, None): (15, 359),
               (3, 1, 1, None): (1, 623), (100, 3, 1, None): (12, 202), (10000, 1, 1, None): (30, 268),
               (100, 3, 624, 1): (2, 487), (10000, 3, 624, 1): (18, 6), (500, 30, 624, 15): (31, 296)}


def find_start(n, count, end_pos, after=None):
    """A (key, start position) from which `count` calls of choice(n, ., replace=False) leave numpy's stream at `end_pos`
    (624: the last draw was word 623 of a block; 1: it was word 0).  `after`: the condition holds after that many of the
    calls instead of after the last one.  choice(n, B) consumes the same draws for every B (a shuffle of arange(n)).

    Keys are random_key(seed) for seed = s0, s0 + 1, ...; start positions 0..624 per key, p0 first, where (s0, p0) is the
    case's entry in START_HINTS: a hit at the first try unless numpy's stream changed (the full search takes up to ~30 s)."""
    k = count if after is None else after
    rs = np.random.RandomState(0)
    seed0, p0 = START_HINTS.get((n, count, end_pos, after), (1, 0))
    for seed in range(seed0, seed0 + 2000):
        key = random_key(seed)
        for p in ([p0] if seed == seed0 else []) + list(range(MT_N + 1)):
            rs.set_state(("MT19937", key, p, 0, 0.0))
            for _ in range(k):
                rs.permutation(n)
            if rs.get_state()[2] == end_pos:
                return key, p
    raise AssertionError("no start position found for n=%d" % n)


# ------------------------------------------------------------------------------------------------ exact sampler: cases
def check_sizes(pkg, n, full_perms):
    """B = 1, 256 and n at one size, from a start position that depends on n; the stream carries over between calls."""
    rb = replay(pkg, n)
    rs = put_state(rb, random_key(n), (n * 7919) % (MT_N + 1))
    draw(rb, rs, 1, 3)
    draw(rb, rs, min(256, n), 2)
    draw(rb, rs, n, full_perms)


def check_update_count(pkg, n, B, count=150):
    assert count * n < 1 << 30
    rb = replay(pkg, n)
    rs = put_state(rb, random_key(n + 1), MT_N)
    draw(rb, rs, B, count)
    draw(rb, rs, B, 1)


def check_start(pkg, n, B, pos):
    rb = replay(pkg, n)
    rs = put_state(rb, random_key(7 * n + pos), pos)
    draw(rb, rs, B, 2)
    draw(rb, rs, B, 1)


def check_block_end(pkg, n, B, count, end_pos=MT_N):
    """The call ends on the last (end_pos 624) or the first (end_pos 1) word of a block; the next call starts there."""
    rb = replay(pkg, n)
    rs = put_state(rb, *find_start(n, count, end_pos))
    assert draw(rb, rs, B, count) == end_pos
    draw(rb, rs, B, 2)                              # from 624: the device must twist the block before its first draw


def check_block_end_inside(pkg, n, B):
    """The first of three samples of one call ends on the last word of a block: the next sample starts on a fresh block."""
    rb = replay(pkg, n)
    key, p = find_start(n, 3, MT_N, after=1)
    rs = put_state(rb, key, p)
    ref = numpy_at(key, p)
    ref.permutation(n)
    assert ref.get_state()[2] == MT_N
    draw(rb, rs, B, 3)


def check_n1_unchanged(pkg):
    """n = 1 draws nothing: a stream at 624 (or anywhere) comes back unchanged, with index 0."""
    rb = replay(pkg, 1)
    key = random_key(1)
    for pos in (MT_N, 0, 311):
        rs = put_state(rb, key, pos)
        assert draw(rb, rs, 1, 4) == pos
        assert np.array_equal(rs.get_state()[1], key)


SIZES = [1, 2, 16383, 16384, 16385, 32767, 32768, 32769, 40000, 55999, 56000]


@pytest.mark.parametrize("n", SIZES)
def test_exact_sampler_sizes_up_to_the_limit(pkg, n):
    check_sizes(pkg, n, 2 if n <= 32769 else 1)


@pytest.mark.parametrize("n,B", [(10000, 100), (MAX_N, 256)])
def test_exact_sampler_150_draws_of_an_update(pkg, n, B):
    check_update_count(pkg, n, B)


@pytest.mark.parametrize("pos", [0, 1, 623, 624])
@pytest.mark.parametrize("n,B", [(2, 1), (3, 3), (97, 5), (10000, 100), (MAX_N, 256)])
def test_exact_sampler_start_positions(pkg, n, B, pos):
    check_start(pkg, n, B, pos)


@pytest.mark.parametrize("n,B,count", [(2, 1, 1), (3, 2, 1), (100, 7, 3), (4097, 256, 1), (10000, 100, 2), (32769, 1, 1),
                                       (MAX_N, 256, 1)])
def test_exact_sampler_ends_on_the_last_word_of_a_block(pkg, n, B, count):
    check_block_end(pkg, n, B, count, MT_N)


@pytest.mark.parametrize("n,B,count", [(3, 2, 1), (100, 7, 3), (10000, 100, 1)])
def test_exact_sampler_ends_on_the_first_word_of_a_block(pkg, n, B, count):
    check_block_end(pkg, n, B, count, 1)


@pytest.mark.parametrize("n,B", [(100, 7), (10000, 256)])
def test_exact_sampler_sample_inside_a_call_ends_on_a_block(pkg, n, B):
    check_block_end_inside(pkg, n, B)


def test_exact_sampler_n1_leaves_the_stream_unchanged(pkg):
    check_n1_unchanged(pkg)


# ------------------------------------------------------------------------------------------------ multi-stream bank, C ABI
def test_exact_sampler_multi_stream_bank_through_the_c_abi(pkg):
    """stream_id k of a bank of five: the drawn stream follows numpy, the other four stay bit-identical, and no stream's cached
    Gaussian (has_gauss, gauss) is touched."""
    L = pkg._lib.lib()
    bank = pkg.MtBank(5, "cuda").seed(np.array([11, 0x5eed, 3, 0xFFFFFFFF, 12345]))
    rss = [np.random.RandomState(int(s)) for s in (11, 0x5eed, 3, 0xFFFFFFFF, 12345)]
    bank.has_gauss.copy_(torch.tensor([1, 0, 1, 1, 0], dtype=torch.int32))
    bank.gauss.copy_(torch.tensor([0.125, -0.0, -1.5, 3e-300, 0.0], dtype=torch.float64))
    for k in range(5):
        assert_stream(bank, k, rss[k])
    for rnd, sid in enumerate([0, 2, 4, 2, 0, 4]):
        n, B, count = 3001 + 1000 * sid + rnd, 37 + rnd, 1 + rnd % 3
        out = torch.empty((count, B), dtype=torch.int32, device="cuda")
        scratch = torch.empty((count * n,), dtype=torch.int32, device="cuda")
        before = [t.clone() for t in (bank.mt, bank.pos, bank.has_gauss, bank.gauss)]
        pkg._lib.check(L.rtd3_sample_indices_mt19937(bank.ref, sid, n, B, count, pkg._lib.ptr(out), pkg._lib.ptr(scratch),
                                                      pkg._lib.stream_ptr()), "sample_indices_mt19937")
        exp = np.stack([rss[sid].choice(n, B, replace=False) for _ in range(count)])
        assert np.array_equal(out.cpu().numpy(), exp)
        assert_stream(bank, sid, rss[sid])
        others = [k for k in range(5) if k != sid]
        assert torch.equal(bank.mt[:, others], before[0][:, others]) and torch.equal(bank.pos[others], before[1][others])
        assert torch.equal(bank.has_gauss, before[2]) and torch.equal(bank.gauss.view(torch.int64), before[3].view(torch.int64))


# ------------------------------------------------------------------------------------------------ numpy's global stream
def numpy_global_at(key, pos, has_gauss=0, gauss=0.0):
    np.random.set_state(("MT19937", np.asarray(key, np.uint32), int(pos), int(has_gauss), float(gauss)))
    return numpy_at(key, pos, has_gauss, gauss)


def assert_global_is(rs):
    g, r = np.random.get_state(), rs.get_state()
    assert g[0] == r[0] and np.array_equal(g[1], r[1]) and g[2] == r[2], "numpy's global stream differs"
    assert g[3] == r[3] and np.float64(g[4]).view(np.int64) == np.float64(r[4]).view(np.int64), "cached Gaussian differs"


def labelled_replay(pkg, n, capacity):
    """Unseeded (numpy's global stream, like the reference); row k holds state (k, k)."""
    rb = pkg.ReplayBuffer(capacity)
    k = torch.arange(n, dtype=torch.float32, device="cuda")
    rb.push(torch.stack([k, k], 1), torch.stack([k, -k], 1), k, torch.stack([k, k], 1), torch.zeros(n, dtype=torch.bool, device="cuda"))
    return rb


@pytest.mark.parametrize("pos,has_gauss", [(624, 0), (0, 1), (623, 1), (311, 0)])
def test_unseeded_sample_follows_numpy_global_stream(pkg, pos, has_gauss):
    saved = np.random.get_state()
    try:
        rb = labelled_replay(pkg, 700, 1000)
        rs = numpy_global_at(random_key(pos), pos, has_gauss, -0.7853981633974483 if has_gauss else 0.0)
        s, a, r, s2, d = rb.sample(64)
        assert np.array_equal(s[:, 0], rs.choice(700, 64, replace=False).astype(np.float32))
        assert_global_is(rs)
        idx = rb.sample_indices(100, 150).cpu().numpy()
        assert np.array_equal(idx, np.stack([rs.choice(700, 100, replace=False) for _ in range(150)]))
        assert_global_is(rs)
        assert np.random.normal() == rs.normal()                          # the cached Gaussian (if any) is the next normal
    finally:
        np.random.set_state(saved)


def test_unseeded_sample_after_an_odd_number_of_normals(pkg):
    saved = np.random.get_state()
    try:
        rb = labelled_replay(pkg, 300, 300)
        np.random.seed(2024)
        rs = np.random.RandomState(2024)
        for _ in range(3):
            assert np.random.normal() == rs.normal()
        assert np.random.get_state()[3] == 1
        s, _, _, _, _ = rb.sample(300)
        assert np.array_equal(s[:, 0], rs.choice(300, 300, replace=False).astype(np.float32))
        assert_global_is(rs)
    finally:
        np.random.set_state(saved)


def test_pipelined_update_with_a_chunk_ending_on_a_block(pkg):
    """td3_update in chunks of 10 epochs (15 index sets each, drawn on the side stream while the previous chunk trains), from a
    numpy state where the first chunk's draw ends on word 623 of a block and a Gaussian is cached: the second chunk's draw
    starts with a twist, and numpy's global stream ends where 30 choice calls leave it, cached Gaussian included."""
    saved = np.random.get_state()
    try:
        n, B, E = 500, 37, 20
        rb = labelled_replay(pkg, n, 1000)
        agent = pkg.TD3(pkg.Residual_Actor_Network(64, 1), pkg.Residual_Critic_Network(64, 1), pkg.Residual_Critic_Network(64, 1),
                        batch_size=B)
        agent.num_epochs, agent.sample_chunk_epochs = E, 10
        per_chunk = 10 + 5                                                  # 10 critic + 5 actor sets (policy delay 2)
        key, p = find_start(n, 2 * per_chunk, MT_N, after=per_chunk)
        rs = numpy_global_at(key, p, 1, 0.3183098861837907)
        agent.td3_update(rb)
        assert agent._side_stream is not None                              # the pipelined path ran
        for c in range(2):
            for _ in range(per_chunk):
                rs.choice(n, B, replace=False)
            if c == 0:
                assert rs.get_state()[2] == MT_N                            # the first chunk ended on the block boundary
        assert_global_is(rs)
    finally:
        np.random.set_state(saved)


# ------------------------------------------------------------------------------------------------ Philox sampler
_M = np.uint64(0xFFFFFFFF)


def philox4x32_10_np(c0, c1, seed):
    """oracle/philox.philox4x32_10 for counters (c0, c1, 0, 0) (uint64 arrays holding 32-bit words) and one 64-bit key."""
    c0, c1 = c0.astype(np.uint64), c1.astype(np.uint64)
    c2, c3 = np.zeros_like(c0), np.zeros_like(c0)
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    m0, m1, w0, w1 = np.uint64(philox.M0), np.uint64(philox.M1), np.uint64(philox.W0), np.uint64(philox.W1)
    s = np.uint64(32)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2                                           # < 2^64: no wrap
        c0, c1, c2, c3 = (p1 >> s) ^ c1 ^ k0, p1 & _M, (p0 >> s) ^ c3 ^ k1, p0 & _M
        k0, k1 = (k0 + w0) & _M, (k1 + w1) & _M
    return c0, c1, c2, c3


def philox_indices(seed, offset, n, B, count):
    """out[4t + k] = (r_k * n) >> 32, r = Philox4x32-10((c lo, c hi, 0, 0), (seed lo, seed hi)), c = offset + t."""
    total = B * count
    c = np.arange((total + 3) // 4, dtype=np.uint64) + np.uint64(offset)
    r = philox4x32_10_np(c & _M, c >> np.uint64(32), seed)
    words = np.stack(r, 1).reshape(-1)[:total]
    return ((words * np.uint64(n)) >> np.uint64(32)).astype(np.int32).reshape(count, B)


def test_philox_restatement_matches_the_oracle():
    rs = np.random.RandomState(4)
    for seed in (0, 0x5eed, (1 << 32) + 5, (1 << 64) - 1, int(rs.randint(0, 1 << 62))):
        ctr = np.concatenate([rs.randint(0, 1 << 62, 12, dtype=np.int64).astype(np.uint64), np.array([0, (1 << 32) - 1, 1 << 32,
                                                                                                        (1 << 64) - 1], np.uint64)])
        got = philox4x32_10_np(ctr & _M, ctr >> np.uint64(32), seed)
        for i, c in enumerate(ctr.tolist()):
            exp = philox.philox4x32_10((c & 0xFFFFFFFF, c >> 32, 0, 0), (seed & 0xFFFFFFFF, seed >> 32))
            assert tuple(int(w[i]) for w in got) == exp


@pytest.mark.parametrize("seed", [0, 0x5eed, (1 << 32) + 5, (1 << 64) - 1])
def test_philox_sampler_bit_for_bit(pkg, seed):
    L = pkg._lib.lib()
    for offset in (0, (1 << 32) - 2):                                      # the second carries into the counter's high word
        for n in (1, 7, 56001, (1 << 31) - 1):
            for B, count in ((5, 3), (1, 1), (256, 9), (1023, 2)):         # count * B mostly not a multiple of 4
                out = torch.full((count, B), -1, dtype=torch.int32, device="cuda")
                pkg._lib.check(L.rtd3_sample_indices_philox(seed, offset, n, B, count, pkg._lib.ptr(out), pkg._lib.stream_ptr()),
                               "sample_indices_philox")
                assert np.array_equal(out.cpu().numpy(), philox_indices(seed, offset, n, B, count)), (seed, offset, n, B, count)


def test_philox_replay_buffer_never_reuses_a_counter(pkg):
    rb = replay(pkg, 70001, seed=987654321)
    rb.sampler = "philox"
    offset = 0
    for B, count in ((5, 3), (7, 1), (256, 150), (3, 3)):
        got = rb.sample_indices(B, count).cpu().numpy()
        assert np.array_equal(got, philox_indices(987654321, offset, 70001, B, count)), (B, count, offset)
        offset += math.ceil(B * count / 4)                                 # 15 draws take counters 0..3, the next call starts at 4
        assert rb._philox_offset == offset


def test_philox_td3_update_draws_once(pkg):
    """An update on the Philox sampler draws its E + n_actor index sets in one call: the offset advances by exactly
    ceil((E + n_actor) * B / 4), and the sets are the oracle's."""
    n, B, E = 3000, 37, 20
    rb = replay(pkg, n, seed=77)
    rb.sampler = "philox"
    rb.sample_indices(3, 1)                                                # the update starts at offset 1
    off0 = rb._philox_offset
    agent = pkg.TD3(pkg.Residual_Actor_Network(64, 1), pkg.Residual_Critic_Network(64, 1), pkg.Residual_Critic_Network(64, 1), batch_size=B)
    agent.num_epochs = E
    agent.td3_update(rb)
    count = E + len(range(0, E, agent.policy_update_delay))               # 20 critic + 10 actor sets: 1 110 draws
    off1 = off0 + math.ceil(count * B / 4)
    assert rb._philox_offset == off1
    used = [st["idx"] for st in agent._graphs.values() if tuple(st["idx"].shape) == (count, B)]
    assert len(used) == 1 and np.array_equal(used[0].cpu().numpy(), philox_indices(77, off0, n, B, count))
    assert np.array_equal(rb.sample_indices(5, 1).cpu().numpy(), philox_indices(77, off1, n, 5, 1))

