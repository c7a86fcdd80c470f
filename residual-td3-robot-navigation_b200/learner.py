"""Replay ring and residual-TD3 learner of the reference (robot.py:58-398) on one B200.

Same names and call surface as the reference:
    ReplayBuffer(capacity).push / sample / __len__                                   robot.py:58-124
    Residual_Actor_Network(), Residual_Critic_Network()  (.layer_1 ... .output_layer) robot.py:128-206
    TD3(actor, critic1, critic2, ...).td3_update / train_critic / train_actor / soft_update
                                                                                     robot.py:209-398
All arithmetic runs in csrc/librtd3.so; torch tensors only own the memory.  The replay rows live in a
device-side SoA ring; a TD3 update draws its 150 minibatch index sets with the numpy-legacy MT19937
protocol on the device (bit-exact with `np.random.choice(len, B, replace=False)`).
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib, constants
from .rng import MtBank

# robot.py:36, 46-54
BUFFER_SIZE = 10000
ACTOR_LR = 0.00001
CRITIC_LR = 0.00001
POLICY_UPDATE_DELAY = 2
TARGET_POLICY_NOISE = 0.2
NOISE_CLIP = 0.5
TD3_EPOCHS = 100
TD3_BATCH_SIZE = 100
GAMMA = 0.99
TAU = 0.001

_COMMS = {}                          # (process group id, device) -> rtd3_comm handle (see TD3._setup_comm)
# "p2p": rtd3_p2p_allreduce, the peer-memory kernel (validated on 2, 4 and 8 B200 of one NVSwitch box: 8 GPUs, B = 256 per rank,
# 107 us per data-parallel epoch against 129 us - profiles/r2_dp_8gpu.md);
# "nccl": rtd3_allreduce_grads on our own NCCL communicator (any topology NCCL serves).  Both are part of the update's CUDA graph.
DEFAULT_DP_COLLECTIVE = "p2p"

HIDDEN = 200     # robot.py:145-148
LAYERS = 3

NET_ACTOR, NET_CRITIC1, NET_CRITIC2, NET_T_ACTOR, NET_T_CRITIC1, NET_T_CRITIC2 = range(6)


def _device(device):
    if not torch.cuda.is_available():
        raise RuntimeError("the learner needs a CUDA device (B200); there is no CPU path")
    return torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)


# ------------------------------------------------------------------------------------------------ replay ring
class ReplayBuffer:
    """robot.py:58-124 as a device ring: s,a,s2 `[cap,2]`, r, notdone `[cap]` float32 (36 B per row)."""

    def __init__(self, capacity, device=None, seed=None):
        self.capacity = int(capacity)
        self.device = _device(device)
        c = self.capacity
        self.s = torch.zeros((c, 2), dtype=torch.float32, device=self.device)
        self.a = torch.zeros((c, 2), dtype=torch.float32, device=self.device)
        self.r = torch.zeros((c,), dtype=torch.float32, device=self.device)
        self.s2 = torch.zeros((c, 2), dtype=torch.float32, device=self.device)
        self.notdone = torch.ones((c,), dtype=torch.float32, device=self.device)
        # rows ever pushed: host mirror + device counter (the device one is authoritative after masked pushes, see
        # Robot.process_transition(types=...): the number of rows those add is only known on the device)
        self._total_host = 0
        self._total_dev = torch.zeros((1,), dtype=torch.int64, device=self.device)
        self._host_stale = False
        self.sampler = "mt19937"      # "mt19937": numpy-exact index draws; "philox": throughput mode (with replacement)
        self._philox_seed = 0x5eed if seed is None else int(seed)
        self._philox_offset = 0
        # index draws come from numpy's global legacy stream (like the reference) unless a seed is given
        self._bank = MtBank(1, self.device)
        self._numpy_global = seed is None
        if seed is not None:
            self._bank.seed(seed)
        self._scratch = None
        self._in_session = False

    def _total(self):
        if self._host_stale:
            self._total_host = int(self._total_dev.item())
            self._host_stale = False
        return self._total_host

    @property
    def position(self):
        return self._total() % self.capacity

    @property
    def size(self):
        return min(self.capacity, self._total())

    def __len__(self):
        return self.size

    def _advance(self, n, device_counted=False):
        """n rows were pushed at `position`; device_counted: the kernel already advanced the device counter."""
        self._total_host = self._total() + n
        if not device_counted:
            self._total_dev += n

    def _mark_device_advanced(self):
        self._host_stale = True

    def push(self, state, action, reward, next_state, done):
        """One transition (numpy / python scalars, like the reference) or n transitions (`[n,2]` / `[n]` CUDA tensors)."""
        if isinstance(state, torch.Tensor) and state.dim() == 2:
            n = state.shape[0]
            s, a, s2 = state.t().contiguous().float(), action.t().contiguous().float(), next_state.t().contiguous().float()
            return self.push_planes(s[0], s[1], a[0], a[1], reward.float().contiguous(), s2[0], s2[1],
                                    done.to(torch.uint8).contiguous(), n)
        row = np.concatenate([np.asarray(state, np.float32).reshape(2), np.asarray(action, np.float32).reshape(2),
                              np.asarray([reward], np.float32), np.asarray(next_state, np.float32).reshape(2)])
        t = torch.from_numpy(row).to(self.device)
        d = torch.tensor([1 if done else 0], dtype=torch.uint8, device=self.device)
        self.push_planes(t[0:1], t[1:2], t[2:3], t[3:4], t[4:5], t[5:6], t[6:7], d, 1)

    def push_planes(self, sx, sy, ax, ay, reward, nx, ny, done, n):
        """n transitions given as env planes (the layout the env / transition kernels produce)."""
        if n > self.capacity:
            raise ValueError("cannot push more rows than the ring holds in one call")
        _lib.check(_lib.lib().rtd3_replay_push(_lib.ptr(self.s), _lib.ptr(self.a), _lib.ptr(self.r), _lib.ptr(self.s2),
                                               _lib.ptr(self.notdone), self.capacity, self.position, _lib.ptr(sx), _lib.ptr(sy),
                                               _lib.ptr(ax), _lib.ptr(ay), _lib.ptr(reward), _lib.ptr(nx), _lib.ptr(ny),
                                               _lib.ptr(done), n, _lib.stream_ptr(self.device)), "replay_push")
        self._advance(n)

    def sample_indices(self, batch_size, count=1):
        """`count` consecutive `np.random.choice(len, batch_size, replace=False)` draws -> int32 `[count, B]` (device)."""
        if self.size < batch_size:
            return None
        out = torch.empty((count, batch_size), dtype=torch.int32, device=self.device)
        if self.sampler == "philox":
            _lib.check(_lib.lib().rtd3_sample_indices_philox(self._philox_seed, self._philox_offset, self.size, batch_size, count,
                                                             _lib.ptr(out), _lib.stream_ptr(self.device)), "sample_indices_philox")
            self._philox_offset += (count * batch_size + 3) // 4
            return out
        need = count * self.size
        if self._scratch is None or self._scratch.numel() < need:
            self._scratch = torch.empty((need,), dtype=torch.int32, device=self.device)
        scratch = self._scratch
        if self._numpy_global and not self._in_session:
            self._bank.sync_from_numpy()
        _lib.check(_lib.lib().rtd3_sample_indices_mt19937(self._bank.ref, 0, self.size, batch_size, count, _lib.ptr(out),
                                                          _lib.ptr(scratch), _lib.stream_ptr(self.device)), "sample_indices")
        if self._numpy_global and not self._in_session:
            self._bank.sync_to_numpy()
        return out

    def begin_sampling_session(self):
        """Several sample_indices calls in a row (a TD3 update draws its index sets in chunks): mirror numpy's global stream
        into the device bank once at the start and back once at the end instead of around every call."""
        if self._numpy_global:
            self._bank.sync_from_numpy()
        self._in_session = True

    def end_sampling_session(self):
        self._in_session = False
        if self._numpy_global:
            self._bank.sync_to_numpy()

    # ---- checkpoint (checkpoint.py) ----------------------------------------------------------------------------------
    def state_dict(self):
        """The whole state of this ReplayBuffer as CPU tensors and plain values (checkpoint.py; synchronises the device)."""
        from . import checkpoint
        return checkpoint.replay_state(self)

    def load_state_dict(self, sd):
        """Load `sd` (from `state_dict` of a ReplayBuffer of the same configuration) in place; every check runs before anything is
        written (ValueError).  With numpy's global stream, numpy's global state is restored too."""
        from . import checkpoint
        checkpoint.load_state(self, sd)
        return self

    def gather(self, idx):
        B = idx.numel()
        idx = idx.to(device=self.device, dtype=torch.int32).contiguous()
        os_, oa, os2 = (torch.empty((B, 2), dtype=torch.float32, device=self.device) for _ in range(3))
        orw, ond = (torch.empty((B,), dtype=torch.float32, device=self.device) for _ in range(2))
        _lib.check(_lib.lib().rtd3_replay_gather(_lib.ptr(self.s), _lib.ptr(self.a), _lib.ptr(self.r), _lib.ptr(self.s2),
                                                 _lib.ptr(self.notdone), _lib.ptr(idx), B, _lib.ptr(os_), _lib.ptr(oa),
                                                 _lib.ptr(orw), _lib.ptr(os2), _lib.ptr(ond), _lib.stream_ptr(self.device)),
                   "replay_gather")
        return os_, oa, orw, os2, ond

    def sample(self, batch_size, as_torch=False):
        """robot.py:98-115: None when under-filled, else (states, actions, rewards, next_states, dones)."""
        idx = self.sample_indices(batch_size, 1)
        if idx is None:
            return None
        s, a, r, s2, nd = self.gather(idx[0])
        dones = nd < 0.5
        if as_torch:
            return s, a, r, s2, dones
        return tuple(t.cpu().numpy() for t in (s, a, r, s2, dones))


# ------------------------------------------------------------------------------------------------ network objects
def _layer_dims(in_dim, hidden, layers, out_dim):
    dims = [in_dim] + [hidden] * layers + [out_dim]
    return list(zip(dims[:-1], dims[1:]))


class _LayerView:
    def __init__(self, weight, bias):
        self.weight, self.bias = weight, bias
        self.in_features, self.out_features = weight.shape[1], weight.shape[0]


class _Network:
    """A network whose parameters are either its own CPU init (before TD3 adopts it) or views of the TD3 arena."""
    in_dim = out_dim = None

    def __init__(self, hidden=HIDDEN, layers=LAYERS):
        self.hidden, self.layers = int(hidden), int(layers)
        # Same torch RNG consumption as the reference constructor: nn.Linear's own init for every layer, then
        # kaiming_uniform_(fan_in, relu) on every weight and zero biases (robot.py:145-151, 161-165).
        lin = [torch.nn.Linear(i, o) for i, o in _layer_dims(self.in_dim, self.hidden, self.layers, self.out_dim)]
        with torch.no_grad():
            for m in lin:
                torch.nn.init.kaiming_uniform_(m.weight, mode="fan_in", nonlinearity="relu")
                torch.nn.init.constant_(m.bias, 0)
        self._flat = torch.cat([torch.cat([m.weight.detach().reshape(-1), m.bias.detach().reshape(-1)]) for m in lin])
        self._td3 = None
        self._net = None
        self._bind_views()

    def count(self):
        return sum(i * o + o for i, o in _layer_dims(self.in_dim, self.hidden, self.layers, self.out_dim))

    def _bind_views(self):
        self._layers = []
        off = 0
        for i, o in _layer_dims(self.in_dim, self.hidden, self.layers, self.out_dim):
            w = self._flat[off:off + i * o].view(o, i)
            off += i * o
            b = self._flat[off:off + o]
            off += o
            self._layers.append(_LayerView(w, b))
        for k, lv in enumerate(self._layers[:-1]):
            setattr(self, "layer_%d" % (k + 1), lv)
        self.output_layer = self._layers[-1]

    def _adopt(self, td3, net):
        """Move into slot `net` of `td3`'s arena; afterwards all attributes are views of device memory."""
        view = td3.flat(net)
        view.copy_(self._flat.to(view.device))
        self._flat, self._td3, self._net = view, td3, net
        self._bind_views()

    @classmethod
    def _view_of(cls, td3, net, hidden, layers):
        obj = cls.__new__(cls)
        obj.hidden, obj.layers = hidden, layers
        obj._flat, obj._td3, obj._net = td3.flat(net), td3, net
        obj._bind_views()
        return obj

    def parameters(self):
        for lv in self._layers:
            yield lv.weight
            yield lv.bias

    def flat_parameters(self):
        return self._flat

    def load_flat(self, values):
        self._flat.copy_(torch.as_tensor(np.asarray(values, dtype=np.float32)).to(self._flat.device))
        if self._td3 is not None:
            self._td3._t_stale = True

    def eval(self):
        return self

    def train(self, mode=True):
        return self


class Residual_Actor_Network(_Network):
    """robot.py:128-165: 2 -> H -> H -> H -> 2, ReLU, linear head."""
    in_dim, out_dim = 2, 2

    def forward(self, input):
        return self._td3.forward(self._net, input)

    __call__ = forward


class Residual_Critic_Network(_Network):
    """robot.py:168-206: cat(state, action) 4 -> H -> H -> H -> 1."""
    in_dim, out_dim = 4, 1

    def forward(self, state, action):
        return self._td3.forward(self._net, torch.cat([state, action], dim=1))

    __call__ = forward


# ------------------------------------------------------------------------------------------------ TD3
class TD3:
    """robot.py:209-398.  `process_group` (torch.distributed, NCCL) makes the learner data-parallel: every rank steps on
    its own replay shard and the flat gradient buffer is all-reduced once per optimiser step."""

    def __init__(self, actor_network, critic_network_1, critic_network_2, actor_lr=ACTOR_LR, critic_lr=CRITIC_LR, gamma=GAMMA,
                 tau=TAU, policy_noise=TARGET_POLICY_NOISE, noise_clip=NOISE_CLIP, policy_update_delay=POLICY_UPDATE_DELAY,
                 num_epochs=TD3_EPOCHS, batch_size=TD3_BATCH_SIZE, device=None, process_group=None, dp_collective=None):
        self.device = _device(device)
        self.hidden, self.layers = actor_network.hidden, actor_network.layers
        for net in (critic_network_1, critic_network_2):
            if (net.hidden, net.layers) != (self.hidden, self.layers):
                raise ValueError("actor and critics must share hidden width and depth")
        self._handle = ctypes.c_void_p()
        _lib.check(_lib.lib().rtd3_td3_create(ctypes.byref(self._handle), self.device.index or 0, self.hidden, self.layers), "td3_create")
        L = _lib.lib()
        self._off = [int(L.rtd3_td3_param_offset(self._handle, k)) for k in range(6)]
        self._cnt = [int(L.rtd3_td3_param_count(self._handle, k)) for k in range(6)]
        total = int(L.rtd3_td3_arena_floats(self._handle))
        self.params = torch.zeros((total,), dtype=torch.float32, device=self.device)
        self.params_t = torch.zeros((total,), dtype=torch.float32, device=self.device)   # hidden weights transposed (forward layout)
        self._t_stale = True
        # "fp32": every product in fp32 FFMA (the parity path).  "tf32": forward passes of >= 128 rows, and critic / actor steps
        # of >= `tc_min_batch` rows (2 x 128 or 2 x 256 networks), run on the tcgen05 tensor cores with TF32 operands (throughput
        # mode; ~1e-3 relative on the outputs).
        self.precision = "fp32"
        self.tc_min_batch = 1024
        self.params_u = None                # [u | v]: tensor-core operand copies of the arena, 2 x total floats
        self.grads = torch.zeros((total // 2,), dtype=torch.float32, device=self.device)
        self.adam_m = torch.zeros_like(self.grads)
        self.adam_v = torch.zeros_like(self.grads)
        self.steps = torch.zeros((2,), dtype=torch.int32, device=self.device)       # Adam step counters {actor, critics}
        self.beta_pows = torch.ones((4,), dtype=torch.float64, device=self.device)  # {0.9^t, 0.999^t} per optimiser
        self._scratch = None
        self._scratch_retired = []

        # online networks adopt arena slots 0..2; targets are copies (copy.deepcopy, robot.py:232-234)
        self.actor_network, self.critic_network_1, self.critic_network_2 = actor_network, critic_network_1, critic_network_2
        actor_network._adopt(self, NET_ACTOR)
        critic_network_1._adopt(self, NET_CRITIC1)
        critic_network_2._adopt(self, NET_CRITIC2)
        half = total // 2
        self.params[half:].copy_(self.params[:half])
        self.target_actor = Residual_Actor_Network._view_of(self, NET_T_ACTOR, self.hidden, self.layers)
        self.target_critic_network_1 = Residual_Critic_Network._view_of(self, NET_T_CRITIC1, self.hidden, self.layers)
        self.target_critic_network_2 = Residual_Critic_Network._view_of(self, NET_T_CRITIC2, self.hidden, self.layers)

        self.actor_lr, self.critic_lr = actor_lr, critic_lr
        self.gamma, self.tau = gamma, tau
        self.policy_noise, self.noise_clip = policy_noise, noise_clip
        self.policy_update_delay = policy_update_delay
        self.max_action = constants.ROBOT_MAX_ACTION
        self.num_epochs, self.batch_size = num_epochs, batch_size
        self.actor_losses, self.critic_losses = [], []
        self.process_group = process_group
        self.world = 1
        if process_group is not None:
            import torch.distributed as dist
            self.world = dist.get_world_size(process_group)
        self.last_losses = None
        self._u_stale = True
        self.params_h = None                # fp16 copies of the hidden weights (rtd3_mlp_forward_f16), built on first use
        self._h_stale = True
        self._side_stream = None
        self.sample_chunk_epochs = 10       # epochs per pipelined chunk of td3_update (0 = draw all index sets up front)
        self._graphs = {}
        self._p2p = None
        self._comm = None
        # target-policy smoothing noise (robot.py:338, torch.randn_like - unseeded in the reference): generated inside the critic
        # kernels from Philox4x32-10 keyed (noise_seed, device step counter, batch row) unless a noise tensor is injected
        self.noise_seed = 0x7d3
        self._noise_counter = torch.zeros((1,), dtype=torch.int64, device=self.device)
        self._noise_steps = 0               # host mirror of the counter (what the next single-step call uses)
        if self.world > 1:                  # initialise the communicator outside of any graph capture
            import torch.distributed as dist
            dist.all_reduce(self.grads, group=process_group)
            self.grads.zero_()
            # Replicas must START identical: every rank drew its initial weights from its own CPU torch generator (unseeded in
            # the reference, robot.py:164), so rank 0's networks are broadcast and the targets re-copied from them (robot.py:232-234).
            # Adam moments, step counters and beta powers are zeros / ones on every rank by construction.
            dist.broadcast(self.params[:half], group=process_group, group_src=0)
            self.params[half:].copy_(self.params[:half])
            self._t_stale = self._u_stale = self._h_stale = True
            import os
            dp_collective = dp_collective or os.environ.get("RTD3_DP_COLLECTIVE", DEFAULT_DP_COLLECTIVE)
            self.dp_collective = dp_collective
            if dp_collective == "p2p":
                self._setup_p2p()
            elif dp_collective == "nccl":
                self._setup_comm()
            else:
                raise ValueError("dp_collective must be 'nccl' or 'p2p'")

    def _setup_comm(self):
        """Our own NCCL communicator behind the C ABI (`rtd3_comm_create`; the unique id travels once over the process group):
        `rtd3_allreduce_grads` on it is a plain stream operation, so the data-parallel update is captured in ONE CUDA graph, NCCL
        node included (torch's ProcessGroupNCCL collectives are not capturable together with foreign launches on this stack)."""
        import torch.distributed as dist
        pg = self.process_group
        rank = dist.get_rank(pg)
        # ONE communicator per (process group, device) for the life of the process, shared by every learner built on it: creating
        # and destroying communicators is itself collective, and Python finalises learners at unpredictable, rank-dependent points
        key = (id(pg), self.device.index or 0)
        if key in _COMMS:
            self._comm = _COMMS[key]
            return
        ident = [None]
        if rank == 0:
            buf = (ctypes.c_uint8 * _lib.COMM_ID_BYTES)()
            _lib.check(_lib.lib().rtd3_comm_unique_id(buf), "comm_unique_id")
            ident = [bytes(buf)]
        dist.broadcast_object_list(ident, group=pg, group_src=0)
        buf = (ctypes.c_uint8 * _lib.COMM_ID_BYTES).from_buffer_copy(ident[0])
        self._comm = ctypes.c_void_p()
        torch.cuda.synchronize(self.device)
        _lib.check(_lib.lib().rtd3_comm_create(ctypes.byref(self._comm), buf, rank, self.world, self.device.index or 0), "comm_create")
        _COMMS[key] = self._comm
        # first collective outside of any capture (connection set-up allocates)
        _lib.check(_lib.lib().rtd3_allreduce_grads(self._comm, _lib.ptr(self.grads), self.grads.numel(), _lib.stream_ptr(self.device)),
                   "allreduce_grads (warm-up)")
        torch.cuda.synchronize(self.device)
        self.grads.zero_()

    def _setup_p2p(self):
        """Gradient all-reduce over NVLink peer memory (`rtd3_p2p_allreduce`): a receive area + flag array per rank that every
        peer maps through CUDA IPC (the handles travel once over the process group); the step kernels keep writing `self.grads`,
        the optimiser kernel consumes the private sum `self._grads_sum`."""
        import ctypes
        import torch.distributed as dist
        from torch.multiprocessing.reductions import reduce_tensor
        pg, world = self.process_group, self.world
        rank = dist.get_rank(pg)
        if world > 8:
            raise ValueError("the peer-memory all-reduce serves up to 8 ranks (one NVSwitch box)")
        G = self.grads.numel()
        S = 2 * G           # floats per slot: a gradient slice in the line form of the fused weight-gradient exchange ({value, step} pairs)
        # receive slots [2][world][S] | flags: uint64 [16] per rank (rtd3_p2p_allreduce) + [8][256] per (rank, block) (the fused all-reduce
        # + optimiser of rtd3_td3_update)
        buf = torch.zeros((2 * world * S + 2 * (16 + 8 * 256),), dtype=torch.float32, device=self.device)
        torch.cuda.synchronize(self.device)
        handles = [None] * world
        dist.all_gather_object(handles, reduce_tensor(buf), group=pg)
        peers = []
        for q in range(world):
            if q == rank:
                peers.append(buf)
                continue
            fn, args = handles[q]
            args = list(args)
            args[6] = self.device.index                 # open the peer's handle in THIS device's context: a P2P mapping
            peers.append(fn(*args))
        self._grads_sum = torch.zeros((G,), dtype=torch.float32, device=self.device)
        c = ctypes.c_void_p * world
        self._p2p = {"peers": peers, "rank": rank, "seq": torch.zeros((1,), dtype=torch.int64, device=self.device), "count": G, "slot": S,
                     "recv": c(*[t.data_ptr() for t in peers]), "flags": c(*[t.data_ptr() + 4 * 2 * world * S for t in peers]),
                     "counter": torch.zeros((1,), dtype=torch.int32, device=self.device)}
        p = self._p2p
        p["struct"] = _lib.P2pStateStruct(ctypes.cast(p["recv"], ctypes.c_void_p), ctypes.cast(p["flags"], ctypes.c_void_p), rank, world,
                                          p["seq"].data_ptr(), self._grads_sum.data_ptr(), S, p["counter"].data_ptr())
        torch.cuda.synchronize(self.device)
        dist.barrier(group=pg)                          # every rank has mapped every buffer before the first launch

    def replica_checksum(self):
        """Order-independent exact checksums of the learner state (int64 sums of the float32 bit patterns of the parameter arena
        and the Adam moments, plus the step counters) -> int64 `[4]` device tensor.  Data-parallel replicas that received the same
        reduced gradients hold bit-identical state, so MIN and MAX of this over the ranks agree (`trainer.replicas_identical`)."""
        bits = lambda t: t.view(torch.int32).to(torch.int64).sum()
        return torch.stack([bits(self.params), bits(self.adam_m), bits(self.adam_v), self.steps.to(torch.int64).sum()])

    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                _lib.lib().rtd3_td3_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    # ---- checkpoint (checkpoint.py) ----------------------------------------------------------------------------------
    def state_dict(self):
        """The whole state of this TD3 as CPU tensors and plain values (checkpoint.py; synchronises the device)."""
        from . import checkpoint
        return checkpoint.td3_state(self)

    def load_state_dict(self, sd):
        """Load `sd` (from `state_dict` of a TD3 of the same configuration) in place; every check runs before anything is
        written (ValueError).  With numpy's global stream, numpy's global state is restored too."""
        from . import checkpoint
        checkpoint.load_state(self, sd)
        return self

    def export_networks(self):
        """The six networks (online and target) as `nn.Module` state dicts keyed by the reference's attribute names (robot.py:232-234):
        {"actor_network": {"layer_1.weight": ..., "output_layer.bias": ...}, ...}, CPU float32.  Loads into modules whose `nn.Linear`
        layers carry the names of robot.py:145-148."""
        from . import checkpoint
        return checkpoint.export_networks(self)

    def import_networks(self, d):
        """Inverse of `export_networks` (bit-exact round trip); checks everything before writing (ValueError)."""
        from . import checkpoint
        checkpoint.import_networks(self, d)

    # ---- arena access ---------------------------------------------------------------------------------
    def flat(self, net):
        """Flat torch-order view of network `net`'s parameters.  Handing it out marks the transposed copy stale (it may be
        written through); edits through previously obtained views need an explicit `sync_transposed()`."""
        self._t_stale = True
        return self.params[self._off[net]:self._off[net] + self._cnt[net]]

    def sync_transposed(self, force=True):
        if force or self._t_stale:
            _lib.check(_lib.lib().rtd3_td3_sync_transposed(self._handle, _lib.ptr(self.params), _lib.ptr(self.params_t),
                                                           _lib.stream_ptr(self.device)), "td3_sync_transposed")
            self._t_stale = False
            self._u_stale = True
            self._h_stale = True

    def _tc_mode(self):
        """"tf32" and "f16" both select the tensor-core paths; they differ in the forward kernel only."""
        return self.precision in ("tf32", "f16")

    def _tc_ok(self, batch):
        return self._tc_mode() and self.hidden % 32 == 0 and 64 <= self.hidden <= 256 and self.layers >= 2 and batch >= 128

    def _f16_ok(self, batch):
        return self.precision == "f16" and self.layers == 2 and self._tc_ok(batch)

    def _sync_half(self, force=False):
        """fp16 copies of the hidden weights for the resident-weight forward; rebuilt whenever the parameters may have changed
        (the optimiser steps mark them stale, and `td3_update` rebuilds them before it returns so that a captured tick graph,
        which cannot run this bookkeeping, always reads current weights)."""
        if self.params_h is None:
            self.params_h = torch.zeros((6 * max(1, self.layers - 1) * self.hidden * self.hidden,), dtype=torch.float16, device=self.device)
            self._h_stale = True
        if force or self._h_stale:
            _lib.check(_lib.lib().rtd3_tc_sync_weights_f16(self.hidden, self.layers, _lib.ptr(self.params), _lib.ptr(self.params_h),
                                                           _lib.stream_ptr(self.device)), "tc_sync_weights_f16")
            self._h_stale = False

    def prepare_forward(self, batch):
        """Bring every derived weight copy the forward of `batch` rows reads up to date (call before capturing a graph that
        contains forwards: the capture must not record these one-off rebuilds)."""
        self.sync_transposed(force=False)
        if self._f16_ok(batch):
            self._sync_half()
        elif self._tc_ok(batch):
            self._sync_chunk_major()

    def _sync_chunk_major(self):
        """Chunk-major weight copy for the tensor-core forward; rebuilt whenever the parameters may have changed (the
        optimiser steps mark it stale)."""
        if self.params_u is None:
            self.params_u = torch.zeros((2 * self.params.numel(),), dtype=torch.float32, device=self.device)
            self._u_stale = True
        if self._u_stale:
            _lib.check(_lib.lib().rtd3_tc_sync_weights(self.hidden, self.layers, _lib.ptr(self.params), _lib.ptr(self.params_u),
                                                       _lib.stream_ptr(self.device)), "tc_sync_weights")
            self._u_stale = False

    def _tc_learner_ok(self, batch):
        return (self._tc_mode() and batch >= self.tc_min_batch
                and bool(_lib.lib().rtd3_td3_tf32_supported(self._handle)))

    def flat_grad(self, net):
        return self.grads[self._off[net]:self._off[net] + self._cnt[net]]

    def forward(self, net, x, select=None):
        """Forward of arena network `net` on `x` `[B,in]` (CUDA float32) -> `[B,out]`.  The kernel (f16, TF32 or fp32) is the one
        the precision selects for `select` rows (default B); each kernel's output rows do not depend on B, so `select` = N on a
        stack of E batches of N rows gives, batch by batch, what the forward of N rows gives."""
        x = x.to(device=self.device, dtype=torch.float32).contiguous()
        out_dim = 2 if net in (NET_ACTOR, NET_T_ACTOR) else 1
        y = torch.empty((x.shape[0], out_dim), dtype=torch.float32, device=self.device)
        rows = x.shape[0] if select is None else int(select)
        self.sync_transposed(force=False)
        if self._f16_ok(rows):
            self._sync_half()
            _lib.check(_lib.lib().rtd3_mlp_forward_f16(self.hidden, self.layers, net, _lib.ptr(self.params), _lib.ptr(self.params_h), _lib.ptr(x),
                                                       _lib.ptr(y), x.shape[0], _lib.stream_ptr(self.device)), "mlp_forward_f16")
            return y
        if self._tc_ok(rows):
            self._sync_chunk_major()
            _lib.check(_lib.lib().rtd3_mlp_forward_tf32(self.hidden, self.layers, 1 if net in (NET_ACTOR, NET_T_ACTOR) else 0, self._off[net],
                                                        _lib.ptr(self.params), _lib.ptr(self.params_u), _lib.ptr(x), _lib.ptr(y), x.shape[0],
                                                        _lib.stream_ptr(self.device)), "mlp_forward_tf32")
            return y
        _lib.check(_lib.lib().rtd3_mlp_forward(self._handle, net, _lib.ptr(self.params), _lib.ptr(self.params_t), _lib.ptr(x), _lib.ptr(y), x.shape[0],
                                               _lib.stream_ptr(self.device)), "mlp_forward")
        return y

    # ---- the three device steps -------------------------------------------------------------------------
    def _grad_range(self, nets):
        """(offset, count) of the gradient floats of the critics (nets = 0b110) or the actor (0b001) in the flat buffer."""
        return (self._off[1], self.grads.numel() - self._off[1]) if nets == 0b110 else (0, self._off[1])

    def _allreduce(self, nets):
        """SUM over the ranks of the gradients one optimiser step consumes (SURVEY.md 8e)."""
        if self.world == 1:
            return
        off, count = self._grad_range(nets)
        if self._p2p is not None:
            p = self._p2p
            _lib.check(_lib.lib().rtd3_p2p_allreduce(p["recv"], p["flags"], p["rank"], self.world, _lib.ptr(p["seq"]), _lib.ptr(self._grads_sum[off:]),
                                                     _lib.ptr(self.grads[off:]), count, p["slot"], _lib.ptr(p["counter"]), _lib.stream_ptr(self.device)),
                       "p2p_allreduce")
        else:
            _lib.check(_lib.lib().rtd3_allreduce_grads(self._comm, _lib.ptr(self.grads[off:]), count, _lib.stream_ptr(self.device)), "allreduce_grads")

    def _row_scratch(self, B):
        need = int(_lib.lib().rtd3_td3_scratch_floats(self._handle, B))
        if self._scratch is None or self._scratch.numel() < need:
            if self._scratch is not None:
                self._scratch_retired.append(self._scratch)    # captured graphs (update and tick graphs) hold its address: never freed
            self._scratch = torch.empty((need,), dtype=torch.float32, device=self.device)
        return self._scratch

    def _critic_step(self, rb, idx, noise, loss2, q_out=None, y_out=None, apply=True):
        """Gradients of both critics into `grads`; `apply` = all-reduce + Adam (False leaves the raw gradients, for tests)."""
        B = idx.numel()
        if self._tc_learner_ok(B):
            self._sync_chunk_major()
            _lib.check(_lib.lib().rtd3_td3_critic_step_tf32(
                self._handle, _lib.ptr(self.params), _lib.ptr(self.params_u), _lib.ptr(self.grads), _lib.ptr(rb.s), _lib.ptr(rb.a),
                _lib.ptr(rb.r), _lib.ptr(rb.s2), _lib.ptr(rb.notdone), _lib.ptr(idx), _lib.ptr(noise), B, self.gamma, self.policy_noise,
                self.noise_clip, float(self.max_action), _lib.ptr(loss2), _lib.ptr(q_out), _lib.ptr(y_out), _lib.ptr(self.steps),
                _lib.ptr(self.beta_pows), _lib.stream_ptr(self.device)), "td3_critic_step_tf32")
            if apply:
                self._allreduce(0b110)
                self._adam(nets=0b110, polyak=0)
            return
        _lib.check(_lib.lib().rtd3_td3_critic_step(
            self._handle, _lib.ptr(self.params), _lib.ptr(self.params_t), _lib.ptr(self.grads), _lib.ptr(self._row_scratch(B)), _lib.ptr(rb.s), _lib.ptr(rb.a),
            _lib.ptr(rb.r), _lib.ptr(rb.s2), _lib.ptr(rb.notdone), _lib.ptr(idx), _lib.ptr(noise), B, self.gamma, self.policy_noise,
            self.noise_clip, float(self.max_action), _lib.ptr(loss2), _lib.ptr(q_out), _lib.ptr(y_out), _lib.ptr(self.steps),
            _lib.ptr(self.beta_pows), _lib.stream_ptr(self.device)), "td3_critic_step")
        if apply:
            self._allreduce(0b110)
            self._adam(nets=0b110, polyak=0)

    def _actor_step(self, rb, idx, loss1):
        B = idx.numel()
        if self._tc_learner_ok(B):
            self._sync_chunk_major()
            _lib.check(_lib.lib().rtd3_td3_actor_step_tf32(self._handle, _lib.ptr(self.params), _lib.ptr(self.params_u), _lib.ptr(self.grads),
                                                           _lib.ptr(rb.s), _lib.ptr(idx), B, _lib.ptr(loss1), _lib.ptr(self.steps),
                                                           _lib.ptr(self.beta_pows), _lib.stream_ptr(self.device)), "td3_actor_step_tf32")
            self._allreduce(0b001)
            return
        _lib.check(_lib.lib().rtd3_td3_actor_step(self._handle, _lib.ptr(self.params), _lib.ptr(self.params_t), _lib.ptr(self.grads),
                                                  _lib.ptr(self._row_scratch(B)), _lib.ptr(rb.s), _lib.ptr(idx), B, _lib.ptr(loss1),
                                                  _lib.ptr(self.steps), _lib.ptr(self.beta_pows), _lib.stream_ptr(self.device)),
                   "td3_actor_step")
        self._allreduce(0b001)

    def _adam(self, nets, polyak):
        # the optimiser kernel keeps the tensor-core copies in step once they exist and are current
        keep_uv = self.params_u is not None and not self._u_stale
        if not keep_uv:
            self._u_stale = True
        self._h_stale = True
        _lib.check(_lib.lib().rtd3_td3_adam_polyak(self._handle, _lib.ptr(self.params), _lib.ptr(self.params_t),
                                                   _lib.ptr(self.params_u if keep_uv else None),
                                                   _lib.ptr(self._grads_sum if self._p2p is not None else self.grads), _lib.ptr(self.adam_m),
                                                   _lib.ptr(self.adam_v), _lib.ptr(self.beta_pows), nets, self.actor_lr, self.critic_lr,
                                                   1.0 / self.world, polyak, self.tau, _lib.stream_ptr(self.device)), "td3_adam_polyak")

    def _noise(self, rows):
        """The unit normals `[rows,2]` the critic kernels would generate for the next step (`rtd3_td3_target_noise`: the same
        Philox4x32-10 stream), for the single-step API; advances the step counter like an update of one epoch does."""
        out = torch.empty((rows, 2), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().rtd3_td3_target_noise(self.noise_seed, self._noise_steps, _lib.ptr(out), rows, _lib.stream_ptr(self.device)),
                   "td3_target_noise")
        self._noise_steps += 1
        self._noise_counter += 1
        return out

    # ---- reference methods --------------------------------------------------------------------------------
    def train_critic(self, replay_buffer, noise=None, idx=None, q_out=None, y_out=None):
        """robot.py:312-366.  `noise` (unit normal `[B,2]`) and `idx` can be injected for parity tests."""
        if idx is None:
            idx = replay_buffer.sample_indices(self.batch_size, 1)
            if idx is None:
                raise TypeError("cannot unpack non-iterable NoneType object")     # what the reference raises when under-filled
            idx = idx[0]
        idx = idx.to(device=self.device, dtype=torch.int32).contiguous()
        noise = self._noise(idx.numel()) if noise is None else noise.to(self.device, torch.float32).contiguous()
        loss2 = torch.zeros((2,), dtype=torch.float32, device=self.device)
        self.sync_transposed(force=False)
        self._critic_step(replay_buffer, idx, noise, loss2, q_out, y_out)
        l = loss2.cpu()
        return float(l[0]), float(l[1])

    def train_actor(self, replay_buffer, idx=None):
        """robot.py:369-398 (the Adam step included; the Polyak updates are td3_update's / soft_update's job)."""
        if idx is None:
            idx = replay_buffer.sample_indices(self.batch_size, 1)
            if idx is None:
                raise TypeError("cannot unpack non-iterable NoneType object")
            idx = idx[0]
        idx = idx.to(device=self.device, dtype=torch.int32).contiguous()
        loss1 = torch.zeros((1,), dtype=torch.float32, device=self.device)
        self.sync_transposed(force=False)
        self._actor_step(replay_buffer, idx, loss1)
        self._adam(nets=0b001, polyak=0)
        return float(loss1.cpu()[0])

    def soft_update(self, target, source, tau):
        """robot.py:293-310 for one (target, source) pair of this agent's networks."""
        pairs = {NET_T_ACTOR: NET_ACTOR, NET_T_CRITIC1: NET_CRITIC1, NET_T_CRITIC2: NET_CRITIC2}
        if getattr(target, "_td3", None) is not self or pairs.get(target._net) != getattr(source, "_net", None):
            raise ValueError("soft_update expects a (target, online) pair of this TD3 agent")
        self.sync_transposed(force=False)
        old_tau, self.tau = self.tau, tau
        try:
            self._adam(nets=0, polyak=1 << (target._net - 3))
        finally:
            self.tau = old_tau

    def _run_epochs(self, rb, idx, noise, closs, aloss):
        """The epoch loop of robot.py:272-285: ONE call of `rtd3_td3_update`, which issues the step kernels, the gradient
        all-reduces and the optimiser kernels on the current stream (capturable in a CUDA graph).  noise None: generated in the
        critic kernels (Philox, keyed by the device step counter, which the call advances)."""
        B = idx.shape[1]
        tc = self._tc_learner_ok(B)
        keep_uv = self.params_u is not None and not self._u_stale
        if tc and not keep_uv:
            raise RuntimeError("tensor-core operand copies are stale: call _sync_chunk_major() first")
        if not keep_uv:
            self._u_stale = True
        self._h_stale = True
        a = _lib.Td3UpdateArgs()
        p = lambda t: None if t is None else t.data_ptr()
        a.params, a.params_t, a.params_uv = p(self.params), p(self.params_t), p(self.params_u if keep_uv else None)
        a.grads, a.adam_m, a.adam_v, a.scratch = p(self.grads), p(self.adam_m), p(self.adam_v), p(None if tc else self._row_scratch(B))
        a.steps, a.beta_pows = p(self.steps), p(self.beta_pows)
        a.rp_s, a.rp_a, a.rp_r, a.rp_s2, a.rp_notdone = p(rb.s), p(rb.a), p(rb.r), p(rb.s2), p(rb.notdone)
        a.idx, a.batch, a.epochs, a.policy_update_delay = p(idx), B, self.num_epochs, self.policy_update_delay
        a.noise, a.noise_seed, a.noise_counter = p(noise), self.noise_seed, p(self._noise_counter)
        a.gamma, a.policy_noise, a.noise_clip, a.max_action = self.gamma, self.policy_noise, self.noise_clip, float(self.max_action)
        a.lr_actor, a.lr_critic, a.tau = self.actor_lr, self.critic_lr, self.tau
        a.critic_losses, a.actor_losses = p(closs), p(aloss)
        a.world, a.tf32 = self.world, 1 if tc else 0
        a.comm = self._comm if (self.world > 1 and self._p2p is None) else None
        if self.world > 1 and self._p2p is not None:
            a.p2p = ctypes.pointer(self._p2p["struct"])
        _lib.check(_lib.lib().rtd3_td3_update(self._handle, ctypes.byref(a), _lib.stream_ptr(self.device)), "td3_update")

    def _coop_ok(self, B):
        # The cooperative single-kernel update was removed (slower than the step kernels at every measured batch,
        # profiles/r2_coop_stage_profile.md); bench.py still asks this to label its TD3 rows.
        return False

    def td3_update(self, replay_buffer, noise=None, idx=None, use_graph=True):
        """robot.py:258-285: `num_epochs` critic steps, an actor step + the three Polyak updates every
        `policy_update_delay`-th epoch.  Returns (critic_losses `[E,2]`, actor_losses `[E_actor]`) as device tensors -
        the values the reference collects at robot.py:274-280.

        The epoch loop is a CUDA graph.  When the index sets are drawn here (idx is None) the update is pipelined in chunks
        of `sample_chunk_epochs` epochs: the exact MT19937 index draw of chunk g+1 runs on a side stream (it needs one SM)
        while chunk g trains, so its cost hides behind the training kernels instead of preceding them."""
        E, B, delay = self.num_epochs, self.batch_size, self.policy_update_delay
        C = self.sample_chunk_epochs
        if (idx is None and use_graph and C > 0 and E % C == 0 and C % delay == 0 and E > C
                and len(replay_buffer) >= B and getattr(replay_buffer, "sampler", "mt19937") == "mt19937"):   # the Philox draw costs microseconds: nothing to hide
            return self._td3_update_pipelined(replay_buffer, noise, C)
        n_actor = len([e for e in range(E) if e % delay == 0])
        count = E + n_actor
        if idx is None:
            idx = replay_buffer.sample_indices(B, count)            # in the order the reference draws them
            if idx is None:
                raise TypeError("cannot unpack non-iterable NoneType object")
        B = idx.shape[1]
        st = self._update_state(replay_buffer, E, B, delay, noise is not None)
        self.sync_transposed(force=False)
        st["idx"].copy_(idx)
        if noise is not None:                                         # injected (parity tests); else generated in the critic kernels
            st["noise"].copy_(noise)
        self._launch_epochs(replay_buffer, st, use_graph, E)
        self.last_losses = (st["closs"], st["aloss"][:n_actor])
        return self.last_losses

    def _update_state(self, replay_buffer, E, B, delay, injected_noise=False):
        """Persistent buffers (and, once captured, the CUDA graph) of an E-epoch block for this replay buffer / batch size."""
        n_actor = len([e for e in range(E) if e % delay == 0])
        key = (id(replay_buffer), E, B, delay, self.precision, self._tc_learner_ok(B), bool(injected_noise))
        st = self._graphs.get(key)
        if st is None:
            st = {"idx": torch.zeros((E + n_actor, B), dtype=torch.int32, device=self.device),
                  "noise": torch.zeros((E, B, 2), dtype=torch.float32, device=self.device) if injected_noise else None,
                  "closs": torch.zeros((E, 2), dtype=torch.float32, device=self.device),
                  "aloss": torch.zeros((max(1, n_actor),), dtype=torch.float32, device=self.device), "graph": None, "launches": 0}
            self._row_scratch(B)
            self._graphs[key] = st
        return st

    def _launch_epochs(self, replay_buffer, st, use_graph, E):
        saved, self.num_epochs = self.num_epochs, E
        tf32 = self._tc_mode()
        if tf32:
            self._sync_chunk_major()         # current before the loop; every optimiser step inside keeps it in step
        try:
            # Both collectives of the data-parallel learner are plain stream operations (our own NCCL communicator, or the
            # peer-memory kernel whose step counter lives in device memory): the update is ONE graph at any world size.
            if use_graph:
                if st["graph"] is None:
                    graph = torch.cuda.CUDAGraph()
                    before = _lib.launch_count()
                    with _lib.capture(graph):
                        self._run_epochs(replay_buffer, st["idx"], st["noise"], st["closs"], st["aloss"])
                    st["graph"] = graph
                    st["launches"] = _lib.launch_count() - before      # kernels inside the graph (capture itself ran none)
                    _lib.lib().rtd3_launch_count_add(-st["launches"])
                st["graph"].replay()
                _lib.lib().rtd3_launch_count_add(st["launches"])
            else:
                self._run_epochs(replay_buffer, st["idx"], st["noise"], st["closs"], st["aloss"])
            if st["noise"] is None:
                self._noise_steps += E       # host mirror of the device step counter the kernels just advanced
        finally:
            self.num_epochs = saved
            if not tf32:
                self._u_stale = True         # a replayed graph does not run _adam's bookkeeping
            self._h_stale = True
            if self.params_h is not None:
                self._sync_half()            # a captured tick graph reads the fp16 copies: current again before the update returns

    def _td3_update_pipelined(self, replay_buffer, noise, C):
        E, B, delay = self.num_epochs, self.batch_size, self.policy_update_delay
        chunks = E // C
        n_actor_c = len([e for e in range(C) if e % delay == 0])
        per_chunk = C + n_actor_c
        st = self._update_state(replay_buffer, C, B, delay, noise is not None)
        closs = torch.empty((E, 2), dtype=torch.float32, device=self.device)
        aloss = torch.empty((chunks * n_actor_c,), dtype=torch.float32, device=self.device)
        self.sync_transposed(force=False)
        main = torch.cuda.current_stream(self.device)
        if self._side_stream is None:
            self._side_stream = torch.cuda.Stream(device=self.device)
        side = self._side_stream
        replay_buffer.begin_sampling_session()                # uploads numpy's stream into the device bank with main-stream kernels ...
        side.wait_stream(main)                                # ... so only now: those writes and the rows pushed so far are visible to the sampler
        try:
            def draw(g):
                with torch.cuda.stream(side):
                    out = replay_buffer.sample_indices(B, per_chunk)
                    ev = torch.cuda.Event()
                    ev.record(side)
                return out, ev
            nxt = draw(0)
            for g in range(chunks):
                idx_g, ev = nxt
                main.wait_event(ev)
                st["idx"].copy_(idx_g)
                if noise is not None:
                    st["noise"].copy_(noise[g * C:(g + 1) * C])
                idx_g.record_stream(main)
                if g + 1 < chunks:
                    nxt = draw(g + 1)                          # runs while chunk g trains (it only touches its scratch and the RNG bank)
                self._launch_epochs(replay_buffer, st, True, C)
                closs[g * C:(g + 1) * C].copy_(st["closs"])
                aloss[g * n_actor_c:(g + 1) * n_actor_c].copy_(st["aloss"][:n_actor_c])
            main.wait_stream(side)
        finally:
            replay_buffer.end_sampling_session()
        self.last_losses = (closs, aloss)
        return self.last_losses
