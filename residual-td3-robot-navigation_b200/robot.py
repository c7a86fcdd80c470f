"""`Robot`: the reference's agent (robot.py:406-823) with its per-step hooks running on the GPU, batched over N envs.

Call surface kept from the reference (SURVEY.md 8b):
    get_next_action_type(state, money) -> 'step' | 'demo' | 'reset'
    get_next_action_training(state, money) -> action      get_next_action_testing(state) -> action
    process_transition(state, action, next_state, money)  process_demonstration(states, actions, money)
    dynamics_model(state, action), attrs goal_state, paths_to_draw, memory (ReplayBuffer), td3_agent (TD3)
`Robot(goal_state)` with a numpy `[2]` goal is the single-env drop-in: numpy in / numpy out, exploration noise and
replay indices drawn from numpy's global legacy stream exactly where the reference draws them.  `Robot(goal_state)`
with a CUDA `[N,2]` goal tensor is the batched form: one shared replay ring and one TD3 agent serve N envs, calls
take / return CUDA tensors, `get_next_action_type` returns an int8 tensor (0 step, 1 demo, 2 reset) and runs one
`td3_update` per `episodes_per_update` finished env-episodes (default N; the reference has no multi-env semantics to copy).
"""
import numpy as np
import torch

from . import _lib, constants
from .learner import (BUFFER_SIZE, ReplayBuffer, Residual_Actor_Network, Residual_Critic_Network, TD3, NET_ACTOR)  # noqa: F401
from .rng import MtBank

# robot.py:22-43
NUM_DEMO = 3
NUM_AUGMENTS = 3
AUG_NOISE = 2.5
AUG_INTERPOLATION = 5
PATH_LENGTH = 50
PATH_INCREASE = 20
INITIAL_NOISE = 1
NOISE_DECAY = 0.75
STUCK_THRESHOLD = 2
STUCK_STEPS = 5
STUCK_PENALTY = 50
GOAL_REWARD = 50
DEMO_PROXIMITY_FACTOR = 10

ACTION_TYPES = ("step", "demo", "reset")
DEMO_GRID, DEMO_CELL = 100, 1.0         # RTD3_DEMO_GRID / RTD3_DEMO_CELL of include/rtd3.h
ENV_DEMO_CELLS = 625                    # RTD3_ENV_DEMO_CELLS

EVAL_MAX_STEPS = 1 << 30                # rtd3_eval_step / rtd3_eval_run_f16 take 1 <= T < 2^30
EVAL_BLOCK_STEPS = 64                   # test steps per captured graph of the per-step evaluation
EVAL_CHECK_BLOCKS = True                # per-step evaluation: read "some env still runs" after each block and end early when none does
EVAL_GRAPHS_KEPT = 4                    # captured evaluation graphs kept per Robot (one per signature)
EVAL_MAX_EPISODES = 1024                # evaluate(episodes=E): 1 <= E <= 1024 and E x N < 2^31 (EVAL_MAX_ROWS), as the kernels take
EVAL_MAX_ROWS = 1 << 31


class PathToDraw:
    """graphics.py:22-30 (pure Python there as well); kept so that `robot.paths_to_draw` has the reference's shape."""

    def __init__(self, path, colour, width):
        self.path = path
        colour = [max(0, min(c, 255)) for c in colour]
        self.line_colour = [int(c) for c in colour]
        self.line_colour.append(255)
        self.line_width = int(width)


def _planes(t, n):
    """[N,2] (any strides) CUDA float32 -> contiguous [2,N]."""
    t = t.to(torch.float32)
    if t.shape == (n, 2):
        t = t.t()
    return t if t.is_contiguous() else t.contiguous()


class Robot:
    def __init__(self, goal_state, hidden=None, layers=None, device=None, seed=None, process_group=None, buffer_size=BUFFER_SIZE,
                 dp_collective=None):
        if not torch.cuda.is_available():
            raise RuntimeError("Robot needs a CUDA device (B200); there is no CPU path")
        self.batched = isinstance(goal_state, torch.Tensor)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.batched:
            g = goal_state.to(self.device, torch.float64)
            self.num_envs = g.shape[0]
            self._goal = (g.t() if g.shape == (self.num_envs, 2) else g).contiguous()        # [2][N]
            self.goal_state = self._goal.t()
        else:
            self.num_envs = 1
            self.goal_state = np.asarray(goal_state, dtype=np.float64)
            self._goal = torch.from_numpy(self.goal_state.reshape(2, 1).copy()).to(self.device)
        n = self.num_envs
        dev = self.device
        self.paths_to_draw = []
        self.demonstration_states = []
        self.demonstration_actions = []
        self._demo_dev = None                                   # [M,2] float64 on the device, the reference's order
        self._demo_cells = None                                 # int32 [DEMO_GRID^2 + 1] offsets into _demo_list, or None: full sweep
        self._demo_list = None                                  # [total,2] float64: per-cell candidate lists (rtd3_demo_lists)
        self.demo_grid_min_points = 64                          # smaller sets are swept in full
        self._env_demo = None                                   # per-env sets (batched process_demonstration), else the shared set above
        # per-env episode state (robot.py:421-438)
        self._num_episodes = torch.zeros(n, dtype=torch.int32, device=dev)
        self._noise_scale = torch.full((n,), float(INITIAL_NOISE), dtype=torch.float64, device=dev)
        self._path_length = torch.full((n,), PATH_LENGTH, dtype=torch.int32, device=dev)
        self._plan_index = torch.zeros(n, dtype=torch.int32, device=dev)
        self._hist = torch.zeros((STUCK_STEPS, 2, n), dtype=torch.float32, device=dev)
        self._hist_count = torch.zeros(n, dtype=torch.int32, device=dev)
        self._hist_head = torch.zeros(n, dtype=torch.int32, device=dev)
        self._goal_reached = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._demo_flag = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._stuck_flag = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._type = torch.zeros(n, dtype=torch.int8, device=dev)
        self._update = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._any_update = torch.zeros(1, dtype=torch.int32, device=dev)
        self._reward = torch.zeros(n, dtype=torch.float32, device=dev)
        self._reward64 = torch.zeros(n, dtype=torch.float64, device=dev)
        self._done = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._base = torch.zeros((n, 2), dtype=torch.float32, device=dev)
        self._action = torch.zeros((2, n), dtype=torch.float32, device=dev)
        self._action64 = torch.zeros((2, n), dtype=torch.float64, device=dev)
        # exploration noise: numpy's global stream for the single-env drop-in, one seeded stream per env otherwise
        self._bank = MtBank(n, dev)
        self._numpy_global = (not self.batched) and seed is None
        if not self._numpy_global:
            self._bank.seed(0 if seed is None else seed)
        self.memory = ReplayBuffer(buffer_size, device=dev, seed=None if self._numpy_global else (0 if seed is None else seed) + 7919)
        kw = {}
        if hidden is not None:
            kw = {"hidden": hidden, "layers": layers if layers is not None else 3}
        self.td3_agent = TD3(actor_network=Residual_Actor_Network(**kw), critic_network_1=Residual_Critic_Network(**kw),
                             critic_network_2=Residual_Critic_Network(**kw), device=dev, process_group=process_group,
                             dp_collective=dp_collective)
        self.num_updates = 0
        self._snap = None
        # One shared learner serves all envs: an update runs once `episodes_per_update` env-episodes have ended since the last
        # one.  The default N keeps the reference's rhythm (every env finishes about one episode between updates) and is
        # exactly the reference for the single-env drop-in (robot.py:480-483).
        self.episodes_per_update = self.num_envs
        self.eval_kernel = True                                 # evaluate() may use rtd3_eval_run_f16 (False: the per-step path)
        self._eval_graphs = {}
        self._eval_work = None

    # ---- reference attributes (single-env views of the device state) --------------------------------------------
    def _scalar(self, t):
        return t[0].item()

    num_episodes = property(lambda self: self._scalar(self._num_episodes) if not self.batched else self._num_episodes)
    current_noise_scale = property(lambda self: self._scalar(self._noise_scale) if not self.batched else self._noise_scale)
    path_length = property(lambda self: self._scalar(self._path_length) if not self.batched else self._path_length)
    plan_index = property(lambda self: self._scalar(self._plan_index) if not self.batched else self._plan_index)
    goal_reached = property(lambda self: bool(self._scalar(self._goal_reached)) if not self.batched else self._goal_reached.bool())
    demo_flag = property(lambda self: bool(self._scalar(self._demo_flag)) if not self.batched else self._demo_flag.bool())
    stuck_flag = property(lambda self: bool(self._scalar(self._stuck_flag)) if not self.batched else self._stuck_flag.bool())

    def _state_planes(self, state):
        if isinstance(state, torch.Tensor):
            return _planes(state.to(self.device), self.num_envs)
        return torch.as_tensor(np.asarray(state, dtype=np.float32).reshape(self.num_envs, 2)).to(self.device).t().contiguous()

    # ---- robot.py:443-506 ------------------------------------------------------------------------------------------
    def advance_action_types(self):
        """Device half of get_next_action_type: the per-env state machine (robot.py:443-489 with reset() :492-506); finished
        episodes are counted into a device counter.  No host synchronisation, so it can sit inside a CUDA graph."""
        _lib.check(_lib.lib().rtd3_robot_next_action_type(
            _lib.ptr(self._num_episodes), _lib.ptr(self._demo_flag), _lib.ptr(self._plan_index), _lib.ptr(self._path_length),
            _lib.ptr(self._goal_reached), _lib.ptr(self._stuck_flag), _lib.ptr(self._noise_scale), _lib.ptr(self._type),
            _lib.ptr(self._update), _lib.ptr(self._any_update), self.num_envs, _lib.stream_ptr(self.device)), "robot_next_action_type")
        return self._type

    def maybe_update(self):
        """Host half: read the finished-episode counter and run td3_update when due (robot.py:480-483).  Synchronous: the host
        waits for the device counter (and, data parallel, for the all-reduce of the ranks' counters)."""
        if self.td3_agent.world > 1:
            from .trainer import update_due
            due = update_due(self._any_update, self.episodes_per_update, self.td3_agent.process_group)
        else:
            due = int(self._any_update.item()) >= self.episodes_per_update
        if due:
            self._any_update.zero_()
            self.td3_agent.td3_update(self.memory)
            self.num_updates += 1
            return True
        return False

    def maybe_update_async(self):
        """`maybe_update` without a host wait on the critical path.  Every call (a) looks at the counter snapshot the PREVIOUS call
        put in flight - by now it has landed in pinned host memory, the device is already running the ticks enqueued since - and
        runs td3_update when `episodes_per_update` (x world) episodes have ended, then (b) puts the next snapshot in flight: the
        device moves the finished-episode counter into a staging word (data parallel: SUM-all-reduced over the ranks, so every rank
        takes the same decision in the same call and enters the update's collectives together) and copies it to the host.
        The decision therefore lags the device by one call (one block of `check_interval` ticks)."""
        agent = self.td3_agent
        if self._snap is None:
            self._snap = {"dev": torch.zeros(1, dtype=torch.int64, device=self.device), "host": torch.zeros(1, dtype=torch.int64).pin_memory(),
                          "event": None, "seen": 0}
        snap = self._snap
        ran = False
        if snap["event"] is not None:
            snap["event"].synchronize()
            snap["seen"] += int(snap["host"][0])
            if snap["seen"] >= self.episodes_per_update * agent.world:
                snap["seen"] = 0
                agent.td3_update(self.memory)
                self.num_updates += 1
                ran = True
        snap["dev"].copy_(self._any_update)
        self._any_update.zero_()
        if agent.world > 1:
            import torch.distributed as dist
            dist.all_reduce(snap["dev"], op=dist.ReduceOp.SUM, group=agent.process_group)
        snap["host"].copy_(snap["dev"], non_blocking=True)
        snap["event"] = torch.cuda.Event()
        snap["event"].record(torch.cuda.current_stream(self.device))
        return ran

    def get_next_action_type(self, state, money_remaining):
        self.advance_action_types()
        self.maybe_update()
        if self.batched:
            return self._type
        return ACTION_TYPES[int(self._type[0].item())]

    def reset(self):
        """robot.py:492-506 applied to every env (the state machine above applies it per env where due)."""
        self._num_episodes += 1
        self._plan_index.zero_()
        self._goal_reached.zero_()
        self._stuck_flag.zero_()
        self._noise_scale *= NOISE_DECAY
        self._path_length += PATH_INCREASE

    # ---- robot.py:509-538 ------------------------------------------------------------------------------------------
    def check_if_stuck(self, state):
        """The reference's stuck test on the PRE-step state, as a stand-alone call (process_transition runs the same logic inside
        `rtd3_robot_transition`, on the same device-side history ring `[5][2][N]`): with five earlier states held and all of them
        closer than STUCK_THRESHOLD the robot is stuck and the history is cleared, otherwise the oldest state is dropped; the
        state is then appended.  Returns a bool (single env) or a bool tensor `[N]`."""
        n = self.num_envs
        sp = self._state_planes(state)                                           # [2,N] float32, what the ring stores
        cnt, head = self._hist_count.long(), self._hist_head.long()
        full = cnt >= STUCK_STEPS
        d = sp.double()[None] - self._hist.double()                               # [5,2,N]
        dist = torch.sqrt(d[:, 1] * d[:, 1] + d[:, 0] * d[:, 0])
        stuck = full & (dist < STUCK_THRESHOLD).all(dim=0)
        head = torch.where(stuck, torch.zeros_like(head), torch.where(full, (head + 1) % STUCK_STEPS, head))
        cnt = torch.where(stuck, torch.zeros_like(cnt), torch.where(full, cnt - 1, cnt))
        slot = (head + cnt) % STUCK_STEPS
        env = torch.arange(n, device=self.device)
        self._hist[slot, 0, env] = sp[0]
        self._hist[slot, 1, env] = sp[1]
        self._hist_count.copy_((cnt + 1).to(torch.int32))
        self._hist_head.copy_(head.to(torch.int32))
        return stuck if self.batched else bool(stuck[0].item())

    # ---- robot.py:541-642 ------------------------------------------------------------------------------------------
    def _act(self, state, noise, types=None):
        n = self.num_envs
        sp = self._state_planes(state)
        L = _lib.lib()
        sptr = _lib.stream_ptr(self.device)
        _lib.check(L.rtd3_robot_baseline(_lib.ptr(sp[0]), _lib.ptr(sp[1]), _lib.ptr(self._goal), _lib.ptr(self._base), n, sptr), "robot_baseline")
        residual = self.td3_agent.forward(NET_ACTOR, self._base)                  # residual_action, robot.py:598-624
        _lib.check(L.rtd3_robot_compose_action(_lib.ptr(sp[0]), _lib.ptr(sp[1]), _lib.ptr(self._goal), _lib.ptr(residual),
                                               _lib.ptr(noise), _lib.ptr(self._noise_scale), _lib.ptr(types), _lib.ptr(self._action[0]),
                                               _lib.ptr(self._action[1]), _lib.ptr(self._action64), n, sptr), "robot_compose_action")
        if self.batched:
            return self._action.t()
        return self._action64[:, 0].cpu().numpy()

    def generate_noise(self, shape=None, types=None):
        """Unit normals `[2,N]` float64 in the order np.random.normal draws them (robot.py:640: x then y per env).  `types` (batched:
        the tick's action types): only the envs whose type is 'step' draw - the reference calls generate_noise on 'step' ticks
        only, so an env's stream advances exactly as its own reference run would."""
        if self._numpy_global:
            self._bank.sync_from_numpy()
        z = self._bank.draw_gauss(2, where=types, equals=0)
        if self._numpy_global:
            self._bank.sync_to_numpy()
        return z

    def get_next_action_training(self, state, money_remaining, noise=None, types=None):
        """`noise`: optional injected unit normals `[2,N]` float64 (tests / throughput mode); default draws them from the
        MT19937 streams.  `types` (batched): the tensor get_next_action_type returned - envs that are not stepping in
        this tick get a null action."""
        z = self.generate_noise(types=types) if noise is None else noise.to(self.device, torch.float64).contiguous()
        return self._act(state, z, types)

    def get_next_action_testing(self, state):
        return self._act(state, None)

    def residual_action(self, state):
        x = torch.as_tensor(np.asarray(state, dtype=np.float32).reshape(-1, 2)).to(self.device) if not isinstance(state, torch.Tensor) else state
        out = self.td3_agent.forward(NET_ACTOR, x)
        return out if self.batched else out[0].cpu().numpy()

    # ---- robot-learning.py:104-117: the test phase, batched ------------------------------------------------------------
    def evaluate(self, environment, max_steps=None, record=False, episodes=None):
        """The reference's test phase for every env i of `environment` (any size and map configuration), with this Robot's
        current actor.  From env i's current state (call `environment.reset()` first for the reference's start), for
        t = 1 .. T (T = `max_steps`, default TEST_TIMEOUT x UPDATE_RATE = 1000): action = get_next_action_testing (no noise)
        against the ENVIRONMENT's goal, step on env i's map, d = |state - goal|; the env stops with success when d <= 5, or at
        t == T.  Returns a dict of CUDA tensors: "success" bool `[N]`, "steps" int32 `[N]` (the step it stopped at),
        "best_distance" float64 `[N]` (smallest d seen) and, with `record`, "trajectory" `[T,N,2]` (a view of `[T,2,N]` planes;
        the rows after an env's stop repeat its final state).  `environment.robot_state` ends at the final states; nothing of
        the Robot changes (only derived weight copies are refreshed, as by any forward).

        `episodes` = E (1 <= E <= 1024, E x N < 2^31): E test episodes of every env in one call, bit-identical to
        `for e in range(E): environment.reset(); r[e] = robot.evaluate(environment, max_steps, record)`.  Episode e of env i
        starts from the (e+1)-th reset draw of env i's stream and runs on env i's map against env i's goal.  The results gain a
        leading episode axis: "success", "steps", "best_distance" `[E,N]`, "start" float32 `[E,N,2]` (each episode's start
        state) and, with `record`, "trajectory" `[E,T,N,2]` (a view of `[E,T,2,N]` float32 planes: E x T x 2 x N x 4 bytes).
        The environment ends where that loop leaves it: the final states of episode E-1, its streams (numpy's global stream
        for a single env without a seed) advanced by E resets, and the last draw as the reset's float64 state.

        With the f16 forward (`precision="f16"`, 2 x H) the whole evaluation, all E episodes included, is one launch
        (`rtd3_eval_run_f16`, `rtd3_eval_run_f16_episodes`); otherwise each step is the actor forward the learner's precision
        selects for N rows (also on the E x N rows of E episodes) plus `rtd3_eval_step` (`rtd3_eval_step_episodes`), replayed
        from CUDA graphs of EVAL_BLOCK_STEPS steps.  Both paths give bit-identical results for the same forward."""
        if max_steps is None:
            T = int(round(constants.TEST_TIMEOUT * constants.UPDATE_RATE))
        else:
            if isinstance(max_steps, bool) or not isinstance(max_steps, (int, np.integer)) or not 1 <= int(max_steps) < EVAL_MAX_STEPS:
                raise ValueError("max_steps must be an integer in [1, 2^30), got %r" % (max_steps,))
            T = int(max_steps)
        E = None
        if episodes is not None:
            if isinstance(episodes, bool) or not isinstance(episodes, (int, np.integer)) or not 1 <= int(episodes) <= EVAL_MAX_EPISODES:
                raise ValueError("episodes must be an integer in [1, %d], got %r" % (EVAL_MAX_EPISODES, episodes))
            E = int(episodes)
        if torch.device(environment.device) != self.device:
            raise ValueError("environment is on %s, the robot on %s" % (environment.device, self.device))
        n = environment.num_envs
        if E is not None and E * n >= EVAL_MAX_ROWS:
            raise ValueError("episodes x num_envs must lie below 2^31, got %d x %d" % (E, n))
        agent = self.td3_agent
        agent.prepare_forward(n)
        dev = self.device
        lead = () if E is None else (E,)
        success = torch.zeros(lead + (n,), dtype=torch.bool, device=dev)
        steps = torch.zeros(lead + (n,), dtype=torch.int32, device=dev)
        best = torch.full(lead + (n,), float("inf"), dtype=torch.float64, device=dev)
        traj = torch.empty(lead + (T, 2, n), dtype=torch.float32, device=dev) if record else None
        starts = None if E is None else torch.empty((E, 2, n), dtype=torch.float32, device=dev)
        if n > 0:
            if self.eval_kernel and agent._f16_ok(n):
                if self._eval_work is None:
                    self._eval_work = torch.zeros(1, dtype=torch.int32, device=dev)
                if E is None:
                    _lib.check(_lib.lib().rtd3_eval_run_f16(
                        environment._handle, agent.hidden, agent.layers, _lib.ptr(agent.params), _lib.ptr(agent.params_h), _lib.ptr(environment._goal),
                        _lib.ptr(environment._state[0]), _lib.ptr(environment._state[1]), _lib.ptr(success), _lib.ptr(steps), _lib.ptr(best),
                        _lib.ptr(traj), 1 if record else 0, n, T, _lib.ptr(self._eval_work), _lib.stream_ptr(dev)), "eval_run_f16")
                else:
                    environment._episode_starts(starts)
                    _lib.check(_lib.lib().rtd3_eval_run_f16_episodes(
                        environment._handle, agent.hidden, agent.layers, _lib.ptr(agent.params), _lib.ptr(agent.params_h), _lib.ptr(environment._goal),
                        _lib.ptr(starts), E, _lib.ptr(environment._state[0]), _lib.ptr(environment._state[1]), _lib.ptr(success), _lib.ptr(steps),
                        _lib.ptr(best), _lib.ptr(traj), 1 if record else 0, n, T, _lib.ptr(self._eval_work), _lib.stream_ptr(dev)), "eval_run_f16_episodes")
            else:
                self._evaluate_steps(environment, T, traj, success, steps, best, starts)
        environment._state_np = None
        out = {"success": success, "steps": steps, "best_distance": best}
        if E is not None:
            out["start"] = starts.permute(0, 2, 1)
        if record:
            out["trajectory"] = traj.transpose(-1, -2)
        return out

    def _evaluate_steps(self, environment, T, traj, success, steps, best, starts=None):
        """The per-step evaluation: the test steps in blocks of S, each block one replay of a captured graph of S (forward,
        `rtd3_eval_step`) pairs.  Envs that have stopped are left alone by the kernel, so the last block may run past T; S is
        chosen so that it runs fewer extra forwards than there are blocks.  With `starts` (`[E,2,N]`, E episodes) the rows are
        the E x N (episode, env) pairs, stepped by `rtd3_eval_step_episodes` on a copy of the start planes drawn here."""
        agent, n, dev = self.td3_agent, environment.num_envs, self.device
        E = None if starts is None else starts.shape[0]
        rows = n if E is None else E * n
        blocks = -(-T // EVAL_BLOCK_STEPS)
        S = -(-T // blocks)
        p = lambda t: None if t is None else t.data_ptr()
        fwd = p(agent.params_h) if agent._f16_ok(n) else (p(agent.params_u) if agent._tc_ok(n) else p(agent.params_t))
        sig = (environment._handle.value, n, E, S, T, agent.precision, p(agent.params), fwd, environment._map_config(), p(environment._state),
               p(environment._goal), p(traj))
        st = self._eval_graphs.get(sig)
        if st is None:
            if len(self._eval_graphs) >= EVAL_GRAPHS_KEPT:
                self._eval_graphs.pop(next(iter(self._eval_graphs)))
            st = {"base": torch.zeros((rows, 2), dtype=torch.float32, device=dev), "success": torch.zeros(rows, dtype=torch.uint8, device=dev),
                  "steps": torch.zeros(rows, dtype=torch.int32, device=dev), "best": torch.zeros(rows, dtype=torch.float64, device=dev)}
            L, x, y = _lib.lib(), environment._state[0], environment._state[1]
            if E is not None:
                st["xs"] = torch.zeros((E, 2, n), dtype=torch.float32, device=dev)

            def step():
                residual = agent.forward(NET_ACTOR, st["base"], select=n)
                if E is None:
                    _lib.check(L.rtd3_eval_step(environment._handle, _lib.ptr(environment._goal), _lib.ptr(x), _lib.ptr(y), _lib.ptr(residual),
                                                _lib.ptr(st["base"]), _lib.ptr(st["success"]), _lib.ptr(st["steps"]), _lib.ptr(st["best"]),
                                                _lib.ptr(traj), 0 if traj is None else 1, n, T, _lib.stream_ptr(dev)), "eval_step")
                else:
                    _lib.check(L.rtd3_eval_step_episodes(environment._handle, _lib.ptr(environment._goal), E, _lib.ptr(st["xs"]), _lib.ptr(residual),
                                                         _lib.ptr(st["base"]), _lib.ptr(st["success"]), _lib.ptr(st["steps"]), _lib.ptr(st["best"]),
                                                         _lib.ptr(traj), 0 if traj is None else 1, n, T, _lib.stream_ptr(dev)), "eval_step_episodes")
            graph = torch.cuda.CUDAGraph()
            before = _lib.launch_count()
            with _lib.capture(graph):
                for _ in range(S):
                    step()
            st["graph"], st["launches"] = graph, _lib.launch_count() - before
            _lib.lib().rtd3_launch_count_add(-st["launches"])
            self._eval_graphs[sig] = st
        st["success"].zero_()
        st["steps"].zero_()
        st["best"].fill_(float("inf"))
        if E is None:
            _lib.check(_lib.lib().rtd3_robot_baseline(_lib.ptr(environment._state[0]), _lib.ptr(environment._state[1]), _lib.ptr(environment._goal),
                                                      _lib.ptr(st["base"]), n, _lib.stream_ptr(dev)), "robot_baseline")
        else:
            environment._episode_starts(starts, st["base"])
            st["xs"].copy_(starts)
        for b in range(blocks):
            st["graph"].replay()
            _lib.lib().rtd3_launch_count_add(st["launches"])
            if EVAL_CHECK_BLOCKS and b + 1 < blocks and not bool(((st["steps"] < T) & (st["success"] == 0)).any()):
                break
        success.view(-1).copy_(st["success"])
        steps.view(-1).copy_(st["steps"])
        best.view(-1).copy_(st["best"])
        if E is not None:
            environment._state.copy_(st["xs"][E - 1])

    # ---- robot.py:645-675 ------------------------------------------------------------------------------------------
    def process_transition(self, state, action, next_state, money_remaining, push=True, types=None):
        n = self.num_envs
        sp, ap, npl = self._state_planes(state), self._state_planes(action), self._state_planes(next_state)
        m = 0 if self._demo_dev is None else self._demo_dev.shape[0]
        rb = self.memory
        d = self._env_demo
        if push and n > rb.capacity:
            raise ValueError("more envs than replay rows: raise buffer_size")
        _lib.check(_lib.lib().rtd3_robot_transition(
            _lib.ptr(self._goal), _lib.ptr(self._hist), _lib.ptr(self._hist_count), _lib.ptr(self._hist_head), _lib.ptr(self._goal_reached),
            _lib.ptr(self._stuck_flag), _lib.ptr(self._demo_flag), _lib.ptr(self._plan_index), _lib.ptr(self._path_length),
            _lib.ptr(sp[0]), _lib.ptr(sp[1]), _lib.ptr(ap[0]), _lib.ptr(ap[1]), _lib.ptr(npl[0]), _lib.ptr(npl[1]),
            _lib.ptr(self._demo_dev), _lib.ptr(self._demo_cells), _lib.ptr(self._demo_list), m, _lib.ptr(self._reward), _lib.ptr(self._reward64), _lib.ptr(self._done),
            _lib.ptr(rb.s if push else None), _lib.ptr(rb.a), _lib.ptr(rb.r), _lib.ptr(rb.s2), _lib.ptr(rb.notdone), rb.capacity,
            0 if types is not None else rb.position, _lib.ptr(rb._total_dev), _lib.ptr(types),
            _lib.ptr(d["sorted"] if d else None), _lib.ptr(d["cells"] if d else None), _lib.ptr(d["count"] if d else None), d["cap"] if d else 0,
            n, _lib.stream_ptr(self.device)),
            "robot_transition")
        if push:
            if types is None:
                rb._advance(n, device_counted=True)
            else:
                rb._mark_device_advanced()              # how many envs stepped is only known on the device

    # ---- robot.py:727-762 (host form, used by process_demonstration; the per-step form lives in the transition kernel) ----
    def compute_reward(self, path):
        goal_distance_reward = -np.linalg.norm(np.asarray(path[-1], dtype=np.float64) - np.asarray(self._goal[:, 0].cpu().numpy()))
        if goal_distance_reward >= -constants.TEST_DISTANCE_THRESHOLD:
            self._goal_reached[0] = 1
            return GOAL_REWARD
        if not self.demonstration_states:
            return goal_distance_reward
        demos = np.asarray(self.demonstration_states, dtype=np.float64)
        mins = [np.sqrt(((demos - np.asarray(step, dtype=np.float64)) ** 2).sum(axis=1)).min() for step in path]
        prox = -np.mean(mins) if bool(self._demo_flag[0].item()) else 0
        return goal_distance_reward + DEMO_PROXIMITY_FACTOR * prox

    # ---- robot.py:679-718, 771-823 (host side: "next" row f-2 of SURVEY.md 8) -------------------------------------------
    def process_demonstration(self, demonstration_states, demonstration_actions, money_remaining):
        if self.batched:
            return self._process_demonstration_batched(demonstration_states, demonstration_actions)
        demonstration_states = np.asarray(demonstration_states)
        demonstration_actions = np.asarray(demonstration_actions)
        self.demonstration_states.extend(demonstration_states)
        self.demonstration_actions.extend(demonstration_actions)
        self.augment_demonstration_data(demonstration_states, demonstration_actions)
        self.draw_path(demonstration_states, colour=[0, 255, 0], width=2)
        self._upload_demos()
        T = len(demonstration_states)
        goal = self._goal[:, 0].cpu().numpy()
        nxt = demonstration_states[1:].astype(np.float64)
        gd = -np.sqrt(((nxt - goal) ** 2).sum(axis=1))
        # compute_reward([next_state]) per transition (robot.py:709-716 -> :727-762): GOAL_REWARD inside the goal radius, else
        # -distance plus - once demo_flag is set, i.e. for a demonstration processed after the demo phase - the proximity term
        # against the demonstration states held NOW (this demonstration and its augmentations included, robot.py:693-697)
        shaped = gd
        if bool(self._demo_flag[0].item()):
            demos = np.asarray([np.asarray(s, dtype=np.float64) for s in self.demonstration_states], dtype=np.float64)
            near = np.array([np.sqrt(((demos - q) ** 2).sum(axis=1)).min() for q in nxt])
            shaped = gd + DEMO_PROXIMITY_FACTOR * (-near)
        rew = np.where(gd >= -constants.TEST_DISTANCE_THRESHOLD, float(GOAL_REWARD), shaped)
        done = np.zeros(T - 1, dtype=bool)
        done[-1] = True
        cu = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(self.device)
        self.memory.push(cu(demonstration_states[:-1]), cu(demonstration_actions[:-1]), cu(rew), cu(demonstration_states[1:]),
                         torch.from_numpy(done).to(self.device))
        self._goal_reached.zero_()                              # robot.py:718

    def _process_demonstration_batched(self, demonstration_states, demonstration_actions):
        """process_demonstration for all N envs (`rtd3_robot_process_demonstration`): `[N,T,2]` float32 CUDA tensors, one
        demonstration per env.  Every env keeps its OWN demonstration set, as every reference run does: the T states and their three
        augmentations (noise from the env's stream, in the reference's draw order) are appended to it, its search grid is rebuilt,
        and the env's T-1 transitions go into the shared replay ring.  From then on the proximity term of env i's reward looks at
        env i's set.  (`demonstration_states` stays a host list only for the single-env form; `demonstration_sets()` reads these.)"""
        n = self.num_envs
        S = demonstration_states.to(self.device, torch.float32).contiguous()
        A = demonstration_actions.to(self.device, torch.float32).contiguous()
        if S.dim() != 3 or S.shape[0] != n or S.shape[2] != 2 or A.shape != S.shape:
            raise ValueError("demonstration_states / demonstration_actions must be [%d,T,2]" % n)
        T = S.shape[1]
        per_demo = T + NUM_AUGMENTS * ((T - 1) * (AUG_INTERPOLATION + 1) + 1)
        if self._env_demo is None:
            cap = NUM_DEMO * per_demo
            self._env_demo = {"cap": cap, "demos": 0,
                              "sets": torch.zeros((n, cap, 2), dtype=torch.float64, device=self.device),
                              "sorted": torch.zeros((n, cap, 2), dtype=torch.float64, device=self.device),
                              "count": torch.zeros((n,), dtype=torch.int32, device=self.device),
                              "cells": torch.zeros((n, ENV_DEMO_CELLS + 1), dtype=torch.int32, device=self.device)}
        d = self._env_demo
        if (d["demos"] + 1) * per_demo > d["cap"]:
            grow = d["cap"] + NUM_DEMO * per_demo
            for k in ("sets", "sorted"):
                big = torch.zeros((n, grow, 2), dtype=torch.float64, device=self.device)
                big[:, :d["cap"]] = d[k]
                d[k] = big
            d["cap"] = grow
        rb = self.memory
        _lib.check(_lib.lib().rtd3_robot_process_demonstration(
            self._bank.ref, _lib.ptr(self._goal), _lib.ptr(self._demo_flag), _lib.ptr(S), _lib.ptr(A), T, _lib.ptr(d["sets"]), _lib.ptr(d["count"]),
            _lib.ptr(d["sorted"]), _lib.ptr(d["cells"]), d["cap"], NUM_AUGMENTS, AUG_INTERPOLATION, float(AUG_NOISE), _lib.ptr(rb.s), _lib.ptr(rb.a),
            _lib.ptr(rb.r), _lib.ptr(rb.s2), _lib.ptr(rb.notdone), rb.capacity, _lib.ptr(rb._total_dev), _lib.stream_ptr(self.device)),
            "robot_process_demonstration")
        d["demos"] += 1
        rb._mark_device_advanced()
        self._goal_reached.zero_()                              # robot.py:718

    def demonstration_sets(self):
        """Batched form: (states `[N,cap,2]` float64 in the reference's append order, counts `[N]`) of the per-env sets, or None."""
        if self._env_demo is None:
            return None
        return self._env_demo["sets"], self._env_demo["count"]

    def set_demonstration_states(self, states):
        """Install a demonstration-state set `[M,2]` directly (batched mode: one set shared by all envs)."""
        self.demonstration_states = list(np.asarray(states, dtype=np.float64))
        self._upload_demos()

    def _upload_demos(self):
        """Demonstration states -> device.  From `demo_grid_min_points` states on, `rtd3_demo_lists` builds the per-cell candidate
        lists that `rtd3_robot_transition` / `rtd3_tick_post` search (robot.py:753's min over ALL demo states, evaluated on the
        handful that can be nearest inside the query's cell); `demonstration_states` itself keeps the reference's order."""
        self._demo_cells = self._demo_list = None
        if not self.demonstration_states:
            self._demo_dev = None
            return
        arr = np.asarray([np.asarray(s, dtype=np.float64) for s in self.demonstration_states], dtype=np.float64)
        self._demo_dev = torch.from_numpy(np.ascontiguousarray(arr)).to(self.device).contiguous()
        m = arr.shape[0]
        if m >= self.demo_grid_min_points:
            L, sp = _lib.lib(), _lib.stream_ptr(self.device)
            cells = DEMO_GRID * DEMO_GRID
            start = torch.zeros(cells + 1, dtype=torch.int32, device=self.device)
            _lib.check(L.rtd3_demo_lists(_lib.ptr(self._demo_dev), m, _lib.ptr(start[1:]), None, None, sp), "demo_lists (count)")
            start[1:] = torch.cumsum(start[1:], 0, dtype=torch.int32)
            total = int(start[-1].item())
            lists = torch.empty((total, 2), dtype=torch.float64, device=self.device)
            _lib.check(L.rtd3_demo_lists(_lib.ptr(self._demo_dev), m, None, _lib.ptr(start), _lib.ptr(lists), sp), "demo_lists (fill)")
            self._demo_cells, self._demo_list = start, lists

    def augment_demonstration_data(self, demonstration_states, demonstration_actions, noise_level=AUG_NOISE,
                                   interpolation_steps=AUG_INTERPOLATION, num_augmentations=NUM_AUGMENTS):
        """robot.py:771-823 with the same numpy draw order (per transition: 5 x (state, action) interpolants, then the
        current (state, action); finally the last (state, action)), vectorised."""
        S, A = np.asarray(demonstration_states), np.asarray(demonstration_actions)
        T = len(S)
        for _ in range(num_augmentations):
            z = np.random.normal(0, noise_level, (T - 1, interpolation_steps + 1, 2, 2))
            zl = np.random.normal(0, noise_level, (2, 2))
            fr = (np.arange(1, interpolation_steps + 1) / float(interpolation_steps + 1)).astype(S.dtype)   # weak python float -> state dtype
            cur, nxt = S[:-1], S[1:]
            synth = cur[:, None, :] + fr[None, :, None] * (nxt - cur)[:, None, :]                       # float32 like the reference
            st = np.concatenate([synth + z[:, :interpolation_steps, 0, :], (cur + z[:, interpolation_steps, 0, :])[:, None, :]], axis=1)
            ac = A[:-1, None, :] + z[:, :, 1, :]
            aug_s = np.concatenate([st.reshape(-1, 2), (S[-1] + zl[0])[None]], axis=0)
            aug_a = np.concatenate([ac.reshape(-1, 2), (A[-1] + zl[1])[None]], axis=0)
            self.draw_path(aug_s, colour=[0, 0, 255], width=2)
            self.demonstration_states.extend(aug_s)
            self.demonstration_actions.extend(aug_a)

    def dynamics_model(self, state, action):
        return state + action                                   # robot.py:722-723

    def draw_path(self, path, colour=[255, 255, 255], width=2):
        self.paths_to_draw.append(PathToDraw(path, colour=colour, width=width))
