"""`Environment`: the reference's world (environment.py:14-183) batched over `num_envs` independent envs on one B200.

Call surface kept from the reference (SURVEY.md section 8b):
    attrs   robot_state, goal_state, robot_init_region ([left,right,bottom,top]), dynamics_speed, dynamics_angle
    methods step(action) -> state, reset() -> state, dynamics(state, action) -> next_state (pure),
            compute_reward(path), get_random_robot_init_state(), set_init_and_goal(), set_dynamics()
With `num_envs == 1` (the default) calls take / return numpy `[2]` float64 arrays like the reference and, unless a
seed is given, draw from numpy's *global* legacy MT19937 stream exactly as the reference does.  With
`num_envs > 1` they take / return CUDA tensors `[N,2]` (views of plane-major `[2,N]` storage, so no copies).

Beyond the reference, the envs of one `Environment` can step on different maps (domain randomisation): `maps` / `set_maps` take a
bank of K maps `[K,100,100]` and `map_index` / `set_map_index` say which map each env uses (`num_maps`, `map_index`).
`map_seeds` / `set_perlin_maps` build such a bank of the reference's own Perlin maps, one per seed, on the device.

All arithmetic happens in csrc/librtd3.so (hand-written sm_100a kernels); there is no CPU path.
"""
import numpy as np
import torch

from . import _lib, configuration, constants
from .rng import MtBank

STEP_AUTO, STEP_SMEM, STEP_LDG = 0, 1, 2


def synthetic_maps(seed=0):
    """Benchmark maps (SURVEY.md 8d, config 2): low-pass filtered uniform noise `u`, speed = sigmoid(10*(u-0.5))
    (the reference's stretch, environment.py:81-83), angle = u; float32 `[100,100]` indexed `[x][y]`.
    `Environment()` without `maps=` builds the reference's own Perlin maps (`perlin_maps`); the benchmarks and parity tests pass
    these instead (the same tensors go to the oracle and to the kernels)."""
    W = constants.WORLD_SIZE
    u = np.random.RandomState(seed).rand(W, W)
    for _ in range(3):
        p = np.pad(u, 1, mode="edge")
        u = (p[1:-1, 1:-1] + p[:-2, 1:-1] + p[2:, 1:-1] + p[1:-1, :-2] + p[1:-1, 2:]) / 5.0
    u = ((u - u.min()) / (u.max() - u.min())).astype(np.float32)
    speed = (1 / (1 + np.exp(-10 * (u - 0.5)))).astype(np.float32)
    return speed, u.copy()


# ---- environment.py:59-95: the reference's own maps ------------------------------------------------------------------------------
# The reference builds them with the third-party `perlin_noise` package (PyPI "perlin-noise", unpinned, not vendored, absent from this
# image): speed = sigmoid-stretched sum of three octaves (5, 10, 20 with weights 1, 0.5, 0.25), angle = one octave (5), both min-max
# normalised, all seeded by configuration.RANDOM_SEED.  PARITY UNPINNED: `_PerlinNoise` restates that package's published algorithm
# (release 1.12: per lattice corner a gradient vector of `random.uniform(-1, 1)` components from Python's generator seeded with
# seed * hasher(corner); corner weight = product of the quintic fade 6t^5 - 15t^4 + 10t^3 of 1 - |distance| per axis; value = sum over
# the cell's corners of weight * dot(gradient, offset)) from its documentation; no reference test or fixture pins the map contents,
# and the maps are INPUTS of the hot path (identical tensors go to the oracle and the kernels).
class _PerlinNoise:
    def __init__(self, octaves=1, seed=1):
        self.octaves, self.seed = octaves, seed
        self._grad = {}

    @staticmethod
    def _fade(t):
        return 6 * t ** 5 - 15 * t ** 4 + 10 * t ** 3

    def _gradient(self, corner):
        g = self._grad.get(corner)
        if g is None:
            import random
            h = max(1, int(abs(sum((10 ** k) * c for k, c in enumerate(corner)) + 1)))
            rnd = random.Random(self.seed * h)
            g = self._grad[corner] = tuple(rnd.uniform(-1, 1) for _ in corner)
        return g

    def __call__(self, coordinates):
        import itertools
        import math
        p = [c * self.octaves for c in coordinates]
        boxes = [(math.floor(c), math.floor(c + 1)) for c in p]
        total = 0.0
        for corner in itertools.product(*boxes):
            d = [a - b for a, b in zip(p, corner)]
            w = 1.0
            for dist in d:
                w *= self._fade(1 - abs(dist))
            total += w * sum(gc * dc for gc, dc in zip(self._gradient(corner), d))
        return total


_PERLIN_CACHE = {}


def perlin_maps(seed=None):
    """`Environment.set_dynamics` (environment.py:59-95) -> (speed, angle) float32 `[100,100]` indexed `[x][y]`; cached per seed (the
    reference seeds the generator with configuration.RANDOM_SEED, so every Environment of a process has the same maps)."""
    seed = configuration.RANDOM_SEED if seed is None else int(seed)
    if seed not in _PERLIN_CACHE:
        W = constants.WORLD_SIZE
        n1, n2, n3 = _PerlinNoise(5, seed), _PerlinNoise(10, seed), _PerlinNoise(20, seed)
        cells = np.zeros([W, W], dtype=np.float32)
        for col in range(W):
            for row in range(W):
                q = [col / W, row / W]
                cells[col, row] = n1(q) + 0.5 * n2(q) + 0.25 * n3(q)
        norm = (cells - np.min(cells)) / (np.max(cells) - np.min(cells))
        speed = 1 / (1 + np.exp(-10 * (norm - 0.5)))                       # stretch_factor 10, environment.py:81-83
        na = _PerlinNoise(5, seed)
        cells = np.zeros([W, W], dtype=np.float32)
        for col in range(W):
            for row in range(W):
                cells[col, row] = na([col / W, row / W])
        angle = (cells - np.min(cells)) / (np.max(cells) - np.min(cells))
        _PERLIN_CACHE[seed] = (speed.astype(np.float32), angle.astype(np.float32))
    s, a = _PERLIN_CACHE[seed]
    return s.copy(), a.copy()


def _checked_seeds(seeds):
    """Seeds of `perlin_maps_device` / `set_perlin_maps` -> int64 CPU tensor `[K]`: a list, a numpy array or an integer tensor on any
    device, 1-D, 1 <= K <= 65536, every value in [0, 2^63); ValueError otherwise.  A CUDA tensor is read back once."""
    if isinstance(seeds, torch.Tensor):
        if seeds.dtype.is_floating_point or seeds.dtype.is_complex or seeds.dtype == torch.bool:
            raise ValueError("map seeds must have an integer dtype, got %s" % seeds.dtype)
        t = seeds.detach().to("cpu")
    else:
        try:
            a = np.asarray(seeds)
        except (OverflowError, ValueError, TypeError) as e:
            raise ValueError("map seeds must be integers in [0, 2^63): %s" % e)
        if a.dtype.kind not in "iu":
            raise ValueError("map seeds must have an integer dtype, got %s" % a.dtype)
        if a.dtype.kind == "u" and a.size and int(a.max()) >= 2 ** 63:
            raise ValueError("map seeds must lie in [0, 2^63)")
        t = torch.from_numpy(a.astype(np.int64))
    if t.dim() != 1 or not 1 <= t.shape[0] <= 65536:
        raise ValueError("map seeds must have shape [K] with 1 <= K <= 65536, got %s" % list(t.shape))
    t = t.to(torch.int64)
    if int(t.min()) < 0:
        raise ValueError("map seeds must lie in [0, 2^63), got %d" % int(t.min()))
    return t.clone()


def _perlin_maps_device(seeds, device):
    """`rtd3_perlin_maps` for checked int64 CPU seeds `[K]` -> (speed, angle) float32 `[K,100,100]` on `device`."""
    W = constants.WORLD_SIZE
    K = seeds.shape[0]
    with torch.cuda.device(device):
        dev_seeds = seeds.to(device)
        speed = torch.empty((K, W, W), dtype=torch.float32, device=device)
        angle = torch.empty((K, W, W), dtype=torch.float32, device=device)
        _lib.check(_lib.lib().rtd3_perlin_maps(_lib.ptr(dev_seeds), K, _lib.ptr(speed), _lib.ptr(angle), _lib.stream_ptr(device)),
                   "perlin_maps")
    return speed, angle


def perlin_maps_device(seeds, device=None):
    """`perlin_maps` for K seeds at once, on the GPU -> (speed, angle) CUDA float32 `[K,100,100]`, map k from `seeds[k]`.
    `seeds`: a list, a numpy array or an integer tensor, 1-D, 1 <= K <= 65536, values in [0, 2^63) (ValueError otherwise).
    `device`: the seeds' CUDA device, else the current one.  `angle` and the fields before normalisation are bit-identical to
    `perlin_maps`; `speed` evaluates exp in float64 rounded once to float32, where numpy uses its host-dependent float32 exp, and
    so differs from `perlin_maps` by a few ulp (include/rtd3.h, rtd3_perlin_maps)."""
    if device is None:
        device = seeds.device if isinstance(seeds, torch.Tensor) and seeds.is_cuda else torch.cuda.current_device()
    return _perlin_maps_device(_checked_seeds(seeds), torch.device(device))


def _planes(t, n, name):
    """[N,2] (any strides) or [2,N] CUDA float32 -> contiguous [2,N] planes; zero-copy when already plane-backed."""
    if t.dim() != 2:
        raise ValueError("%s must be 2-D" % name)
    if t.shape == (n, 2):          # documented layout; for n == 2 a [2,2] tensor is read as [N,2]
        t = t.t()
    elif t.shape != (2, n):
        raise ValueError("%s must have shape [%d,2]" % (name, n))
    if t.dtype != torch.float32:
        t = t.to(torch.float32)
    return t if t.is_contiguous() else t.contiguous()


class Environment:
    def __init__(self, num_envs=1, device=None, seed=None, maps=None, map_index=None, map_seeds=None):
        """`maps`: (speed, angle), each `[100,100]` or a bank `[K,100,100]`; None builds the reference's Perlin maps.
        `map_seeds`: instead of `maps`, a bank of the reference's Perlin maps, one per seed, built on the device (`set_perlin_maps`).
        `map_index`: int `[num_envs]`, the map of every env (see `set_maps`)."""
        if maps is not None and map_seeds is not None:
            raise ValueError("pass maps or map_seeds, not both")
        if not torch.cuda.is_available():
            raise RuntimeError("Environment needs a CUDA device (B200); there is no CPU path")
        self.num_envs = int(num_envs)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        n = self.num_envs
        self._handle = _lib.c_void_p()
        _lib.check(_lib.lib().rtd3_env_create(_lib.ctypes.byref(self._handle), self.device.index or 0), "env_create")
        self._state = torch.zeros((2, n), dtype=torch.float32, device=self.device)        # x plane, y plane
        self._state64 = torch.zeros((2, n), dtype=torch.float64, device=self.device)      # last reset draw (float64)
        self._state_np = None                                                             # single env: cached host copy of the state
        self._goal = torch.zeros((2, n), dtype=torch.float64, device=self.device)
        self._region = torch.zeros((4, n), dtype=torch.float64, device=self.device)       # left,right,bottom,top
        self._bank = MtBank(n, self.device)
        # single env + no seed: mirror numpy's global stream like the reference (robot-learning.py:19-22)
        self._numpy_global = (n == 1 and seed is None)
        if not self._numpy_global:
            self._bank.seed(configuration.RANDOM_SEED if seed is None else seed)
        self.step_variant = STEP_AUTO
        self._pipe = None
        self._pipe_buf = None
        self._map_index = None
        self._map_seeds = None
        self.num_maps = 1
        self.set_init_and_goal()
        if map_seeds is not None:
            self.set_perlin_maps(map_seeds, index=map_index)
        elif maps is None:
            self.set_dynamics()
            if map_index is not None:
                self.set_map_index(map_index)
        else:
            self.set_maps(*maps, index=map_index)

    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                _lib.lib().rtd3_env_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    # ---- checkpoint (checkpoint.py) ----------------------------------------------------------------------------------
    def state_dict(self):
        """The whole state of this Environment as CPU tensors and plain values (checkpoint.py; synchronises the device)."""
        from . import checkpoint
        return checkpoint.env_state(self)

    def load_state_dict(self, sd):
        """Load `sd` (from `state_dict` of a Environment of the same configuration) in place; every check runs before anything is
        written (ValueError).  With numpy's global stream, numpy's global state is restored too."""
        from . import checkpoint
        checkpoint.load_state(self, sd)
        return self

    # ---- RNG plumbing -------------------------------------------------------------------------------
    def _rng_in(self):
        if self._numpy_global:
            self._bank.sync_from_numpy()

    def _rng_out(self):
        if self._numpy_global:
            self._bank.sync_to_numpy()

    # ---- reference attributes -----------------------------------------------------------------------
    @property
    def robot_state(self):
        """Single env: a float64 numpy `[2]` array, the SAME object until the state next changes (the reference returns
        `self.robot_state` itself from `step`, environment.py:127, so `env.step(a) is env.robot_state`).  Batched: the `[N,2]`
        view of the device planes."""
        if self.num_envs == 1:
            if self._state_np is None:
                self._state_np = self._state[:, 0].double().cpu().numpy()
            return self._state_np
        return self._state.t()

    @robot_state.setter
    def robot_state(self, value):
        if self.num_envs == 1 and not isinstance(value, torch.Tensor):
            value = torch.as_tensor(np.asarray(value, dtype=np.float32).reshape(1, 2))
        self._state.copy_(_planes(value.to(self.device), self.num_envs, "robot_state"))
        self._state_np = None

    @property
    def goal_state(self):
        if self.num_envs == 1:
            return self._goal[:, 0].cpu().numpy()
        return self._goal.t()

    @property
    def robot_init_region(self):
        if self.num_envs == 1:
            return self._region[:, 0].cpu().numpy()
        return self._region.t()

    # ---- environment.py:28-56 -----------------------------------------------------------------------
    def set_init_and_goal(self):
        self._rng_in()
        _lib.check(_lib.lib().rtd3_env_init_goal_region(self._bank.ref, _lib.ptr(self._goal), _lib.ptr(self._region),
                                                        _lib.stream_ptr(self.device)), "env_init_goal_region")
        self._rng_out()

    # ---- environment.py:59-95 (map contents are inputs; generator parity is unpinned, see perlin_maps) ------------------
    def set_dynamics(self):
        self.set_maps(*perlin_maps(configuration.RANDOM_SEED))

    def set_maps(self, speed, angle, index=None):
        """Set the dynamics maps: `[100,100]` speed and angle (every env on that map), or a bank of K maps `[K,100,100]`.
        With a bank, env i steps on map `index[i]` (int `[num_envs]`, values in [0, K)); the default index for K > 1 is
        contiguous blocks, `index[i] = i*K // num_envs`: the rollout kernels stage one map per CTA (32 to 256 consecutive envs),
        and warps on their CTA's map run at the single-map speed; other warps read their tables from global memory, several times
        slower.  `dynamics_speed` / `dynamics_angle` are `[K,100,100]` for K > 1 and `[100,100]` otherwise."""
        W = constants.WORLD_SIZE
        speed = torch.as_tensor(np.asarray(speed.cpu() if isinstance(speed, torch.Tensor) else speed, dtype=np.float32))
        angle = torch.as_tensor(np.asarray(angle.cpu() if isinstance(angle, torch.Tensor) else angle, dtype=np.float32))
        if speed.shape != angle.shape or speed.dim() not in (2, 3) or tuple(speed.shape[-2:]) != (W, W) or speed.numel() == 0:
            raise ValueError("maps must be [%d,%d] or [K,%d,%d], speed and angle alike" % (W, W, W, W))
        self._install_maps(speed, angle, index)

    def set_perlin_maps(self, seeds, index=None):
        """`set_maps` with the bank `perlin_maps_device(seeds)`: map k is the reference's Perlin map of `seeds[k]`, generated on the
        device and handed to the library there; only `dynamics_speed` / `dynamics_angle` take one device-to-host copy.  `seeds`: a
        list, a numpy array or an integer tensor, 1-D, 1 <= K <= 65536, values in [0, 2^63) (ValueError otherwise); `index` as in
        `set_maps`.  `map_seeds` holds the seeds until maps are next set another way."""
        seeds = _checked_seeds(seeds)
        self._install_maps(*_perlin_maps_device(seeds, self.device), index, seeds=seeds)

    @property
    def map_seeds(self):
        """int64 `[K]` CPU tensor (a copy) of the seeds the maps were generated from, or None for maps from `maps=`, `set_maps` or
        `set_dynamics`."""
        return None if self._map_seeds is None else self._map_seeds.clone()

    def _install_maps(self, speed, angle, index, seeds=None):
        """Installs float32 maps `[100,100]` or `[K,100,100]` (checked by the caller): CPU tensors are uploaded, CUDA tensors on this
        device go to the library as they are.  Nothing changes when `index` is rejected."""
        K = 1 if speed.dim() == 2 else int(speed.shape[0])
        if speed.dim() == 3 and index is None and K > 1:
            n = self.num_envs
            index = torch.arange(n, dtype=torch.int64) * K // n
        idx = None if index is None else self._checked_index(index, K)
        def host(t):                                       # the numpy attribute: [100,100] for a single map
            t = t[0] if K == 1 and t.dim() == 3 else t
            return t.cpu().numpy() if t.is_cuda else t.numpy().copy()
        self.dynamics_speed = host(speed)
        self.dynamics_angle = host(angle)
        self._speed_dev = speed.contiguous().to(self.device)
        self._angle_dev = angle.contiguous().to(self.device)
        if speed.dim() == 2:
            _lib.check(_lib.lib().rtd3_env_set_map(self._handle, _lib.ptr(self._speed_dev), _lib.ptr(self._angle_dev),
                                                   _lib.stream_ptr(self.device)), "env_set_map")
        else:
            _lib.check(_lib.lib().rtd3_env_set_maps(self._handle, _lib.ptr(self._speed_dev), _lib.ptr(self._angle_dev), K,
                                                    _lib.stream_ptr(self.device)), "env_set_maps")
        self.num_maps = K
        self._map_seeds = seeds
        self._set_index(idx)

    def set_map_index(self, index):
        """Which map of the bank each env steps on: int `[num_envs]` with values in [0, num_maps) (None: every env on map 0).
        Raises ValueError for a non-integer dtype, a wrong length or a value out of range; the range check reads the index's
        minimum and maximum back to the host (one synchronisation per call).  The handle keeps its own copy, written
        asynchronously in place, so a captured CUDA graph replayed afterwards sees the new index.  Rule of every kernel: with
        an index of length m, env (or row) v of a launch steps on map `index[v % m]`."""
        self._set_index(None if index is None else self._checked_index(index, self.num_maps))

    @property
    def map_index(self):
        """int32 `[num_envs]` CUDA tensor (a copy), or None when every env steps on map 0 without an index."""
        return None if self._map_index is None else self._map_index.clone()

    def _checked_index(self, index, K):
        n = self.num_envs
        t = index if isinstance(index, torch.Tensor) else torch.as_tensor(np.asarray(index))
        if t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
            raise ValueError("map index must have an integer dtype, got %s" % t.dtype)
        if t.dim() != 1 or t.shape[0] != n:
            raise ValueError("map index must have shape [%d], got %s" % (n, list(t.shape)))
        t = t.to(self.device)
        lo, hi = torch.stack(torch.aminmax(t)).tolist()   # the one host synchronisation of a set
        if lo < 0 or hi >= K:
            raise ValueError("map index values must lie in [0, %d), got [%d, %d]" % (K, lo, hi))
        return t.to(dtype=torch.int32, copy=True).contiguous()   # our own copy: the caller may reuse theirs

    def _set_index(self, idx):
        self._map_index = idx                              # kept alive: the library copies it asynchronously
        _lib.check(_lib.lib().rtd3_env_set_map_index(self._handle, _lib.ptr(idx), 0 if idx is None else idx.numel(),
                                                     _lib.stream_ptr(self.device)), "env_set_map_index")

    def _map_config(self):
        """(bank address, index address, K, m) as the library's launches capture them (rtd3_env_map_config)."""
        tables, index, K, m = _lib.c_void_p(), _lib.c_void_p(), _lib.c_int32(), _lib.c_int64()
        _lib.check(_lib.lib().rtd3_env_map_config(self._handle, _lib.ctypes.byref(tables), _lib.ctypes.byref(index),
                                                  _lib.ctypes.byref(K), _lib.ctypes.byref(m)), "env_map_config")
        return tables.value, index.value, K.value, m.value

    # ---- environment.py:98-119 ----------------------------------------------------------------------
    def dynamics(self, state, action):
        """Pure next state of n rows; with a map bank row j uses env `j % num_envs`'s map."""
        single = not isinstance(state, torch.Tensor)
        if single:
            s = torch.as_tensor(np.asarray(state, dtype=np.float32).reshape(1, 2)).to(self.device)
            a = torch.as_tensor(np.asarray(action, dtype=np.float32).reshape(1, 2)).to(self.device)
        else:
            s, a = state, action
        n = s.shape[0]
        sp, ap = _planes(s, n, "state"), _planes(a, n, "action")
        out = torch.empty((2, n), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().rtd3_env_dynamics(self._handle, _lib.ptr(sp[0]), _lib.ptr(sp[1]), _lib.ptr(ap[0]),
                                                _lib.ptr(ap[1]), _lib.ptr(out[0]), _lib.ptr(out[1]), n,
                                                _lib.stream_ptr(self.device)), "env_dynamics")
        if single:
            return out[:, 0].double().cpu().numpy()
        return out.t()

    # ---- environment.py:122-127 ---------------------------------------------------------------------
    def step(self, action):
        n = self.num_envs
        if not isinstance(action, torch.Tensor):
            action = torch.as_tensor(np.asarray(action, dtype=np.float32).reshape(n, 2)).to(self.device)
        ap = _planes(action, n, "action")
        _lib.check(_lib.lib().rtd3_env_step(self._handle, _lib.ptr(self._state[0]), _lib.ptr(self._state[1]),
                                            _lib.ptr(ap[0]), _lib.ptr(ap[1]), n, self.step_variant,
                                            _lib.stream_ptr(self.device)), "env_step")
        self._state_np = None
        return self.robot_state

    def rollout(self, actions, record=True):
        """T calls of `step` in one launch.  `actions`: CUDA float32 `[T,N,2]` backed by `[T,2,N]` planes
        (e.g. `planes.permute(0,2,1)`) or a contiguous `[T,2,N]` tensor.  Returns the trajectory `[T,N,2]`
        (a view of `[T,2,N]` planes) if `record`, else None; `robot_state` ends at the final state."""
        n = self.num_envs
        if actions.dim() != 3:
            raise ValueError("actions must be [T,N,2] or [T,2,N]")
        if actions.shape[1:] == (n, 2):
            planes = actions.permute(0, 2, 1)
        else:
            planes = actions
        if planes.shape[1:] != (2, n):
            raise ValueError("actions must be [T,%d,2] or [T,2,%d]" % (n, n))
        if planes.dtype != torch.float32:
            planes = planes.float()
        planes = planes if planes.is_contiguous() else planes.contiguous()
        T = planes.shape[0]
        traj = torch.empty((T, 2, n), dtype=torch.float32, device=self.device) if record else None
        _lib.check(_lib.lib().rtd3_env_rollout(self._handle, _lib.ptr(self._state[0]), _lib.ptr(self._state[1]),
                                               _lib.ptr(planes), _lib.ptr(traj), n, T,
                                               _lib.stream_ptr(self.device)), "env_rollout")
        self._state_np = None
        return traj.permute(0, 2, 1) if record else None

    def rollout_host(self, actions_host, out_host=None, chunks=None, mode=None):
        """`rollout` for HOST buffers: `actions_host` float32 `[T,2,N]` (planes), `out_host` `[T,2,N]` or None.  Pinned buffers
        are mapped into the device's address space (UVA), so the copy engines and the rollout kernel's TMA tiles reach them:

        mode "graph_in" (default for pinned buffers): `rtd3_env_rollout_host` - the T steps in `chunks` (8) time slices, the
            copy engine brings the actions of slice c+1 to HBM while the kernel runs slice c and writes its trajectory tiles
            straight to the host buffer (TMA stores across PCIe); the whole pipeline is ONE CUDA graph cached in the library per
            (buffers, shape), so a call is one graph launch: 0.834 ms per synchronous call for 4096 x 1000 (16 slices 0.846,
            32 slices 0.971: a slice costs ~7 us of hand-over, the first one's copy is exposed);
        mode "graph": both directions through the copy engines (H2D of slice c+1, kernel of slice c, D2H of slice c-1): 0.920 ms
            with 4 slices, 0.943 with 8, 1.07 with 16 - every memcpy node adds ~8 us to the chain;
        mode "graph_out": the kernel reads the host actions itself, the trajectory goes back through the copy engine: 1.22 ms
            (TMA tile reads across PCIe are the slow direction);
        mode "zero_copy": ONE launch; the kernel's TMA tile loads read the actions from host memory and its tile stores write
            the trajectory back, both overlapped with the recurrence, nothing staged in HBM (0.926 ms);
        mode "hybrid": the "graph_in" pipeline issued eagerly from Python on torch streams (0.95 ms);
        mode "staged" (any buffers; the default when one is pageable): the "graph" pipeline issued eagerly from Python on three
            torch streams (0.934 ms).
        For reference, the two raw copies run concurrently take 0.70 ms for these bytes: every mode is PCIe-bound
        (`tools/e2e_graph.py`).

        Returns `out_host` (a fresh pinned tensor if None was given); the call returns once the result is on the host."""
        n = self.num_envs
        if actions_host.dim() != 3 or actions_host.shape[1:] != (2, n) or actions_host.dtype != torch.float32:
            raise ValueError("actions_host must be float32 [T,2,%d]" % n)
        T = actions_host.shape[0]
        if out_host is None:
            out_host = torch.empty((T, 2, n), dtype=torch.float32).pin_memory()
        if out_host.shape != (T, 2, n) or out_host.dtype != torch.float32 or not out_host.is_contiguous() or not actions_host.is_contiguous():
            raise ValueError("out_host must be a contiguous float32 [T,2,%d] like actions_host" % n)
        pinned = actions_host.is_pinned() and out_host.is_pinned()
        if mode is None:
            mode = "graph_in" if pinned else "staged"
        graph_modes = {"graph": 3, "graph_in": 1, "graph_out": 2}
        if mode not in ("hybrid", "zero_copy", "staged") and mode not in graph_modes:
            raise ValueError("mode must be 'graph', 'graph_in', 'graph_out', 'zero_copy', 'hybrid' or 'staged'")
        if mode != "staged" and not pinned:
            raise ValueError("mode %r needs pinned host buffers" % mode)
        main = torch.cuda.current_stream(self.device)
        self._state_np = None
        if mode in graph_modes:
            _lib.check(_lib.lib().rtd3_env_rollout_host(self._handle, _lib.ptr(self._state[0]), _lib.ptr(self._state[1]),
                                                        _lib.ptr(actions_host), _lib.ptr(out_host), n, T,
                                                        8 if chunks is None else int(chunks), graph_modes[mode],
                                                        _lib.stream_ptr(self.device)), "env_rollout_host")
            main.synchronize()
            return out_host
        chunks = 8 if chunks is None else int(chunks)
        if mode == "zero_copy":
            _lib.check(_lib.lib().rtd3_env_rollout(self._handle, _lib.ptr(self._state[0]), _lib.ptr(self._state[1]),
                                                   _lib.ptr(actions_host), _lib.ptr(out_host), n, T,
                                                   _lib.stream_ptr(self.device)), "env_rollout")
            main.synchronize()
            return out_host
        if self._pipe is None:
            self._pipe = (torch.cuda.Stream(device=self.device), torch.cuda.Stream(device=self.device))
        s_in, s_out = self._pipe
        if self._pipe_buf is None or self._pipe_buf[0].shape != (T, 2, n):
            self._pipe_buf = (torch.empty((T, 2, n), dtype=torch.float32, device=self.device),
                              torch.empty((T, 2, n), dtype=torch.float32, device=self.device))
        d_act, d_traj = self._pipe_buf
        s_in.wait_stream(main)
        s_out.wait_stream(main)
        bounds = [round(c * T / chunks) for c in range(chunks + 1)]
        ev_in = []
        for c in range(chunks):
            lo, hi = bounds[c], bounds[c + 1]
            with torch.cuda.stream(s_in):
                d_act[lo:hi].copy_(actions_host[lo:hi], non_blocking=True)
                e = torch.cuda.Event()
                e.record(s_in)
            ev_in.append(e)
        for c in range(chunks):
            lo, hi = bounds[c], bounds[c + 1]
            if hi == lo:
                continue
            main.wait_event(ev_in[c])
            dst = out_host if mode == "hybrid" else d_traj
            _lib.check(_lib.lib().rtd3_env_rollout(self._handle, _lib.ptr(self._state[0]), _lib.ptr(self._state[1]),
                                                   _lib.ptr(d_act[lo:hi]), _lib.ptr(dst[lo:hi]), n, hi - lo,
                                                   _lib.stream_ptr(self.device)), "env_rollout")
            if mode == "hybrid":
                continue
            e = torch.cuda.Event()
            e.record(main)
            with torch.cuda.stream(s_out):
                s_out.wait_event(e)
                out_host[lo:hi].copy_(d_traj[lo:hi], non_blocking=True)
        main.wait_stream(s_out)
        main.synchronize()
        return out_host

    # ---- environment.py:130-137 ---------------------------------------------------------------------
    def reset(self, mask=None, where_equals=None):
        """Redraw the start state inside the fixed init region: all envs, those where `mask` is set, or - `where_equals` given -
        those where the int8 / uint8 tensor `mask` equals that value (the action types of the batched loop go in as they are)."""
        m, eq = None, -1
        if mask is not None:
            if where_equals is not None:
                if mask.dtype not in (torch.int8, torch.uint8):
                    raise TypeError("where_equals needs an int8 / uint8 tensor")
                m, eq = mask.to(self.device).contiguous(), int(where_equals)
            else:
                m = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        self._rng_in()
        _lib.check(_lib.lib().rtd3_env_reset(self._bank.ref, _lib.ptr(self._region), _lib.ptr(m), eq, _lib.ptr(self._state[0]),
                                             _lib.ptr(self._state[1]), _lib.ptr(self._state64),
                                             _lib.stream_ptr(self.device)), "env_reset")
        self._rng_out()
        if self.num_envs == 1:
            # the reference returns the float64 draw itself, and it IS robot_state afterwards (environment.py:131-132); the
            # device keeps its float32 rounding
            self._state_np = self._state64[:, 0].cpu().numpy()
            return self._state_np
        return self.robot_state

    def _episode_starts(self, starts, base=None):
        """E calls of `reset()` in one launch (`rtd3_eval_starts`), for E evaluation episodes: the draws go to `starts`
        `[E,2,N]` float32 instead of the state, the streams advance by E resets and `_state64` holds the last draw.  `base`:
        optional `[E*N,2]` float32 that gets each episode's first actor input, start - goal."""
        self._rng_in()
        _lib.check(_lib.lib().rtd3_eval_starts(self._bank.ref, _lib.ptr(self._region), _lib.ptr(self._goal), starts.shape[0], _lib.ptr(starts),
                                               _lib.ptr(base), _lib.ptr(self._state64), _lib.stream_ptr(self.device)), "eval_starts")
        self._rng_out()

    def get_random_robot_init_state(self):
        """environment.py:135-137: a draw that does not move the robot."""
        keep, keep_np = self._state.clone(), self._state_np
        out = self.reset()
        out = out.copy() if self.num_envs == 1 else out.clone()
        self._state.copy_(keep)
        self._state_np = keep_np
        return out

    # ---- environment.py:140-179 (SURVEY.md 8 row f-1: the 80 000 serial dynamics calls become 4 rollouts of 100 paths) ----
    def get_demonstration(self):
        """Cross-entropy-method planner of the reference.  Random draws (start state, iteration-0 action signs, later
        Gaussian action samples) come from numpy's stream in the reference's order; the 100 x 200-step path rollouts of
        every iteration run as one launch of the rollout kernel (float32 state, so paths agree with the float64
        reference to the per-step tolerance, not bit for bit)."""
        if self.num_envs != 1:
            return self._get_demonstration_batched()
        c = constants
        I, P, T, E = c.DEMOS_CEM_NUM_ITERATIONS, c.DEMOS_CEM_NUM_PATHS, c.DEMOS_CEM_PATH_LENGTH, c.DEMOS_CEM_NUM_ELITES
        planning_actions = np.zeros([I, P, T, 2], dtype=np.float32)
        planning_paths = np.zeros([I, P, T + 1, 2], dtype=np.float32)
        planning_path_rewards = np.zeros([I, P])
        start = self.get_random_robot_init_state()
        goal = self.goal_state
        mean = std = None
        for it in range(I):
            if it == 0:
                acts = np.random.choice([-c.ROBOT_MAX_ACTION, c.ROBOT_MAX_ACTION], (P, T, 2))
            else:
                acts = np.random.normal(mean[None], std[None], (P, T, 2))
            planning_actions[it] = acts
            x = torch.full((P,), float(np.float32(start[0])), dtype=torch.float32, device=self.device)
            y = torch.full((P,), float(np.float32(start[1])), dtype=torch.float32, device=self.device)
            planes = torch.from_numpy(np.ascontiguousarray(planning_actions[it].transpose(1, 2, 0))).to(self.device)   # [T,2,P]
            traj = torch.empty((T, 2, P), dtype=torch.float32, device=self.device)
            _lib.check(_lib.lib().rtd3_env_rollout(self._handle, _lib.ptr(x), _lib.ptr(y), _lib.ptr(planes), _lib.ptr(traj), P, T,
                                                   _lib.stream_ptr(self.device)), "env_rollout")
            planning_paths[it, :, 0] = start
            planning_paths[it, :, 1:] = traj.permute(2, 0, 1).cpu().numpy()
            planning_path_rewards[it] = -np.sqrt(((planning_paths[it, :, -1].astype(np.float64) - goal) ** 2).sum(axis=1))
            elites = np.argsort(planning_path_rewards[it].copy())[-E:]
            mean = np.mean(planning_actions[it, elites], axis=0)
            std = np.std(planning_actions[it, elites], axis=0)
        best = np.argmax(planning_path_rewards[-1])
        return planning_paths[-1, best, 0:T], planning_actions[-1, best]

    def _cem_workspace(self):
        """Device buffers of the batched planner (`rtd3_cem_workspace`), allocated on first use and kept."""
        if getattr(self, "_cem", None) is None:
            c, n, dev = constants, self.num_envs, self.device
            P, T, E = c.DEMOS_CEM_NUM_PATHS, c.DEMOS_CEM_PATH_LENGTH, c.DEMOS_CEM_NUM_ELITES
            f32 = lambda *shape: torch.zeros(shape, dtype=torch.float32, device=dev)
            t = {"actions": f32(T, 2, P * n), "x": f32(P * n), "y": f32(P * n), "start_x": f32(n), "start_y": f32(n),
                 "start64": torch.zeros((2, n), dtype=torch.float64, device=dev), "rewards": torch.zeros((n, P), dtype=torch.float64, device=dev),
                 "elite": torch.zeros((n, E), dtype=torch.int32, device=dev), "best": torch.zeros((n,), dtype=torch.int32, device=dev),
                 "mean": f32(T, 2, n), "std": f32(T, 2, n), "best_actions": f32(T, 2, n), "traj": f32(T, 2, n)}
            w = _lib.CemWorkspaceStruct(*[t[k].data_ptr() for k, _ in _lib.CemWorkspaceStruct._fields_])
            self._cem = (t, w)
        return self._cem

    def _get_demonstration_batched(self, it_begin=0, it_end=None, finish=True):
        """`get_demonstration` for all N envs at once (`rtd3_env_get_demonstration`): every env plans from its own start state to
        its own goal on its own MT19937 stream - the draws and their order are the reference's - and the 100 x N rollouts of an
        iteration are one launch of the rollout kernel.  Returns (states `[N,200,2]`, actions `[N,200,2]`) float32 CUDA tensors.
        `it_begin / it_end / finish` run a part of the planner (tests look at the workspace between iterations)."""
        c, n = constants, self.num_envs
        I, P, T, E = c.DEMOS_CEM_NUM_ITERATIONS, c.DEMOS_CEM_NUM_PATHS, c.DEMOS_CEM_PATH_LENGTH, c.DEMOS_CEM_NUM_ELITES
        t, w = self._cem_workspace()
        states = torch.empty((n, T, 2), dtype=torch.float32, device=self.device) if finish else None
        actions = torch.empty((n, T, 2), dtype=torch.float32, device=self.device) if finish else None
        _lib.check(_lib.lib().rtd3_env_get_demonstration(self._handle, self._bank.ref, _lib.ptr(self._region), _lib.ptr(self._goal),
                                                         _lib.ctypes.byref(w), I, P, T, E, it_begin, I if it_end is None else it_end, 1 if finish else 0,
                                                         _lib.ptr(states), _lib.ptr(actions), _lib.stream_ptr(self.device)), "env_get_demonstration")
        return states, actions

    # ---- environment.py:182-183 ---------------------------------------------------------------------
    def compute_reward(self, path):
        if self.num_envs == 1 and not isinstance(path, torch.Tensor):
            return -np.linalg.norm(np.asarray(path)[-1] - self.goal_state)
        last = path[-1].to(torch.float64)                      # [N,2]
        return -torch.linalg.norm(last - self._goal.t(), dim=1)
