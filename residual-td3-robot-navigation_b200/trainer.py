"""Batched restatement of the training branch of the reference's `update(dt)` (robot-learning.py:66-101), plus the
env-range sharding used for multi-GPU runs (SURVEY.md 8e).

One tick = what the reference does for one env per call of `update`, applied to all N envs of this rank:
    types = robot.get_next_action_type(state, money)          robot-learning.py:68   (runs td3_update when an episode ended)
    type 'reset' -> state = environment.reset()               robot-learning.py:82-85
    type 'step'  -> action = robot.get_next_action_training(state); next = environment.step(action);
                    robot.process_transition(state, action, next); state = next     robot-learning.py:95-101
    type 'demo'  -> batched mode has no per-env planner call yet: the tick is a no-op for that env (demonstration
                    states are installed up front with Robot.set_demonstration_states)
Money accounting keeps the reference's counters per env (demos / resets / steps bought); the wall-clock term
(robot-learning.py:47) is replaced by a fixed per-tick charge so that runs are deterministic.
"""
import torch

from . import constants


def shard_range(num_envs, rank, world):
    """Contiguous env-index range of `rank`: envs are independent, so sharding is a partition with no data-path collective."""
    if num_envs % world != 0:
        raise ValueError("num_envs must divide evenly over the ranks (equal shards keep mean-of-means == global mean)")
    per = num_envs // world
    return rank * per, (rank + 1) * per


def allreduce_grads_(flat_grads, group=None):
    """The one collective of the data-parallel learner: SUM all-reduce of the flat gradient buffer over the ranks
    (NCCL over NVLink on the GPUs; the optimiser kernel then applies the 1/world scale).  Returns the world size."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return 1
    world = dist.get_world_size(group)
    if world > 1:
        dist.all_reduce(flat_grads, op=dist.ReduceOp.SUM, group=group)
    return world


def replicas_identical(td3_agent, group=None):
    """True iff every rank's learner state (parameters incl. targets, Adam moments, step counters) is bit-identical: the exact
    integer checksums of `TD3.replica_checksum` are MIN- and MAX-all-reduced and compared.  Collective: call it on all ranks."""
    import torch.distributed as dist
    c = td3_agent.replica_checksum()
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return True
    lo, hi = c.clone(), c.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
    return bool((lo == hi).all().item())


def update_due(local_count, episodes_per_update, group=None):
    """Whether a learner update is due, decided identically on every rank: the data-parallel `td3_update` all-reduces its
    gradients, so all ranks must enter it in the same tick.  `local_count` (int tensor `[1]`, this rank's finished-episode
    counter) is SUM-all-reduced and compared with `episodes_per_update` x world; with a single rank it is compared directly.
    (A rank-local decision deadlocked the 2-GPU full-loop run: one rank entered the update's all-reduce, the other did not.)"""
    import torch.distributed as dist
    world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
    if world > 1:
        total = local_count.clone()
        dist.all_reduce(total, op=dist.ReduceOp.SUM, group=group)
        return int(total.item()) >= int(episodes_per_update) * world
    return int(local_count.item()) >= int(episodes_per_update)


class DriverLoop:
    """The reference's driver, robot-learning.py:19-117, for ONE env, without pyglet: `update()` is the body of `update(dt)` with the
    script's globals as attributes (`mode, demos_bought, resets_bought, steps_bought, test_best_distance, penalty, state`).  It calls
    the drop-in `Environment` / `Robot` hooks exactly where the script calls the reference's, so with a numpy `[2]` goal the numpy
    global stream is consumed as in the reference.  Two deliberate differences, both for determinism: the wall-clock term of
    `calculate_remaining_money` (robot-learning.py:47) is `ticks x tick_seconds` (default 1/UPDATE_RATE s, the interval the script
    schedules `update` at) instead of `time.time()`, and the test time-out (robot-learning.py:115) is counted in the same ticks;
    `pyglet.app.exit()` becomes `finished = True`."""

    def __init__(self, environment, robot, state=None, tick_seconds=None, verbose=False):
        self.environment, self.robot = environment, robot
        self.state = environment.reset() if state is None else state          # robot-learning.py:22
        self.mode = "training"
        self.demos_bought = self.resets_bought = self.steps_bought = 0
        self.test_ticks = 0
        self.test_best_distance = float("inf")
        self.penalty = False
        self.success = False
        self.finished = False
        self.ticks = 0                                                        # update() calls so far = the deterministic clock
        self.tick_seconds = (1.0 / constants.UPDATE_RATE) if tick_seconds is None else float(tick_seconds)
        self.test_timeout_ticks = max(1, int(round(constants.TEST_TIMEOUT / self.tick_seconds))) if self.tick_seconds > 0 else 1000
        self.verbose = verbose
        self.last_action_type = None

    @classmethod
    def from_seed(cls, seed=None, maps=None, **kw):
        """robot-learning.py:19-24: seed numpy's global stream, build the environment, reset it, build the robot on its goal."""
        import numpy as np
        from . import configuration
        from .environment import Environment
        from .robot import Robot
        np.random.seed(configuration.RANDOM_SEED if seed is None else seed)
        environment = Environment(maps=maps)
        state = environment.reset()
        return cls(environment, Robot(environment.goal_state), state, **kw)

    def _say(self, msg):
        if self.verbose:
            print(msg)

    def calculate_remaining_money(self):
        c = constants
        cpu_time_bought = self.ticks * self.tick_seconds
        money_spent = (self.demos_bought * c.COST_PER_DEMO + self.resets_bought * c.COST_PER_RESET + self.steps_bought * c.COST_PER_STEP
                       + cpu_time_bought * c.COST_PER_CPU_SECOND)
        return c.STARTING_MONEY - money_spent

    def update(self):
        """One call of update(dt) (robot-learning.py:54-117).  Returns the action type of a training tick, 'test' for a test step,
        None once the run is over."""
        import numpy as np
        c = constants
        environment, robot = self.environment, self.robot
        if self.finished:
            return None
        if self.mode == "training":
            money_remaining = self.calculate_remaining_money()
            action_type = robot.get_next_action_type(self.state, money_remaining)
            money_remaining = self.calculate_remaining_money()
            self.ticks += 1
            self.last_action_type = action_type
            if money_remaining < 0:
                if money_remaining < -1.0:
                    self._say("You have overspent by more than 1! A 10% penalty will be applied to the score.")
                    self.penalty = True
                self.state = environment.reset()
                self.mode = "testing"
                self._say("Training has finished, moving to testing.")
                return "switch"
            if action_type == "reset":
                if money_remaining >= c.COST_PER_RESET:
                    self.state = environment.reset()
                    self.resets_bought += 1
                else:
                    self._say("Insufficient money to buy a reset.")
            elif action_type == "demo":
                if money_remaining >= c.COST_PER_DEMO:
                    demonstration_states, demonstration_actions = environment.get_demonstration()
                    robot.process_demonstration(demonstration_states, demonstration_actions, money_remaining)
                    self.demos_bought += 1
                else:
                    self._say("Insufficient money to buy a demo.")
            elif action_type == "step":
                if money_remaining >= c.COST_PER_STEP:
                    action = robot.get_next_action_training(self.state, money_remaining)
                    next_state = environment.step(action)
                    robot.process_transition(self.state, action, next_state, money_remaining)
                    self.state = next_state
                    self.steps_bought += 1
            else:
                raise ValueError("Invalid value for action_type: %s" % (action_type,))
            return action_type
        action = robot.get_next_action_testing(self.state)
        next_state = environment.step(action)
        distance = np.linalg.norm(next_state - environment.goal_state)
        self.state = next_state
        self.test_ticks += 1
        if distance <= c.TEST_DISTANCE_THRESHOLD:
            self._say("The robot reached the goal! Time: %s." % (self.test_ticks * self.tick_seconds,))
            self.success = self.finished = True
        if distance < self.test_best_distance:
            self.test_best_distance = distance
        if self.test_ticks >= self.test_timeout_ticks:
            self._say("The robot did not reach the goal in time. Best distance: %s." % (self.test_best_distance,))
            self.finished = True
        return "test"

    def run(self, max_ticks=None):
        """Call update() until the run is over (or `max_ticks` calls); returns the number of calls made."""
        k = 0
        while not self.finished and (max_ticks is None or k < max_ticks):
            self.update()
            k += 1
        return k


class BatchedTrainer:
    """`graph=True` captures the device work of one tick (state machine, act, step, transition + replay push, masked reset)
    in a CUDA graph and looks at the finished-episode counter only every `check_interval` ticks, so the tick costs one graph
    launch instead of a dozen kernel launches and a device->host read.  With `graph=False, check_interval=1` every tick is
    launched eagerly and checked immediately (the single-env-like behaviour).

    `fused=True` runs the tick as three launches - `rtd3_tick_pre`, the actor forward, `rtd3_tick_post` (csrc/rtd3_tick.cu) -
    instead of one launch per hook; every array ends up bit-identical (tests/test_tick_gpu.py), only the order in which the
    stepping envs' rows land in the replay ring differs (it is atomic-ordered in both forms).  `run(ticks)` with `graph=True`
    replays `check_interval` fused ticks from ONE graph.

    noise: "mt19937" per-env numpy-legacy streams (exact mode); "randn" torch's generator; "philox" (fused only) normals
    generated inside `rtd3_tick_post` from (seed, device tick counter, env)."""

    def __init__(self, environment, robot, noise="mt19937", graph=False, check_interval=1, fused=False, philox_seed=0x5eed,
                 async_check=False, scheduler=False, tick_seconds=None, demonstrations=False):
        if environment.num_envs != robot.num_envs:
            raise ValueError("environment and robot must hold the same envs")
        self.env, self.robot = environment, robot
        self.n = environment.num_envs
        self.device = environment.device
        self.env.reset()
        self.noise = noise                    # "mt19937": per-env numpy-legacy streams; "randn": torch's Philox (throughput mode)
        self.steps_bought = torch.zeros(self.n, dtype=torch.int64, device=self.device)
        self.resets_bought = torch.zeros(self.n, dtype=torch.int64, device=self.device)
        self.ticks = 0
        self.check_interval = max(1, int(check_interval))
        self._prev = torch.empty((2, self.n), dtype=torch.float32, device=self.device)
        self._z = torch.zeros((2, self.n), dtype=torch.float64, device=self.device)
        self._use_graph = bool(graph)
        self._graph = None
        self._graph_k = None
        self.fused = bool(fused)
        if noise == "philox" and not self.fused:
            raise ValueError('noise="philox" is generated inside the fused tick kernel: pass fused=True')
        if noise not in ("mt19937", "randn", "philox"):
            raise ValueError("unknown noise mode %r" % (noise,))
        self.philox_seed = int(philox_seed)
        self.multi_tick_kernel = True         # run() may use rtd3_tick_run_f16 (see _multi_tick_ok)
        # async_check: the "is a learner update due" test never makes the host wait for the device (Robot.maybe_update_async: the
        # decision is taken from the counter snapshot of the previous block); False = the synchronous test after every block
        self.async_check = bool(async_check)
        # demonstrations: a 'demo' tick does what the reference does (robot-learning.py:88-92): every env plans its own
        # demonstration (Environment.get_demonstration, batched CEM) and the robot processes it (per-env demonstration sets,
        # augmentation, replay rows).  All envs request their demonstrations in lock step - ticks 0 .. NUM_DEMO-1 of a run
        # (robot.py:468-470) - so no device -> host read is needed to know when.  False: 'demo' ticks are no-ops and the caller
        # installs a shared set with Robot.set_demonstration_states.
        self.demonstrations = bool(demonstrations)
        self._tick_counter = torch.zeros(2, dtype=torch.int64, device=self.device)      # [ticks completed, scratch of the tick in flight]
        # scheduler: the rest of update(dt) (robot-learning.py:45-50, 66-117) as per-env device state inside the fused tick kernels -
        # money gates on every purchase, demos_bought, the switch to testing once the money is gone, the test branch (success
        # within TEST_DISTANCE_THRESHOLD, best distance, time-out).  The wall-clock term of the money (COST_PER_CPU_SECOND) is
        # charged deterministically: `tick_seconds` per tick (default: the 1/UPDATE_RATE s the reference schedules update(dt) at).
        self.scheduler = bool(scheduler)
        self.tick_seconds = (1.0 / constants.UPDATE_RATE) if tick_seconds is None else float(tick_seconds)
        if self.scheduler:
            if not self.fused:
                raise ValueError("the scheduler lives in the fused tick kernels: pass fused=True (the hook-by-hook form is driven "
                                 "from the host like the reference's update(dt): trainer.DriverLoop)")
            dev = self.device
            self.mode = torch.zeros(self.n, dtype=torch.uint8, device=dev)              # 0 training, 1 testing, 2 finished
            self.demos_bought = torch.zeros(self.n, dtype=torch.int64, device=dev)
            self.test_ticks = torch.zeros(self.n, dtype=torch.int32, device=dev)
            self.test_best_distance = torch.full((self.n,), float("inf"), dtype=torch.float64, device=dev)
            self.test_success = torch.zeros(self.n, dtype=torch.uint8, device=dev)
            self.penalty = torch.zeros(self.n, dtype=torch.uint8, device=dev)
            self.test_timeout_ticks = max(1, int(round(constants.TEST_TIMEOUT / self.tick_seconds))) if self.tick_seconds > 0 else 1000

    def money_remaining(self, tick_charge=None):
        """calculate_remaining_money (robot-learning.py:45-50) per env, float64 `[N]`; the wall-clock term is ticks x tick_charge
        money (default: tick_seconds x COST_PER_CPU_SECOND with the scheduler, else 0)."""
        c = constants
        if tick_charge is None:
            tick_charge = self.tick_seconds * c.COST_PER_CPU_SECOND if self.scheduler else 0.0
        demos = self.demos_bought if self.scheduler else 0
        return (c.STARTING_MONEY - (demos * c.COST_PER_DEMO + self.resets_bought * c.COST_PER_RESET + self.steps_bought.double() * c.COST_PER_STEP
                                    + self.ticks * tick_charge))

    def all_finished(self):
        """Scheduler: every env has finished its test phase (device -> host read)."""
        return self.scheduler and bool((self.mode == 2).all().item())

    def results(self):
        """Scheduler: what the reference prints at the end of a run (robot-learning.py:111, 116), per env, as numpy arrays."""
        if not self.scheduler:
            raise RuntimeError("results() needs scheduler=True")
        f = lambda t: t.cpu().numpy()
        return {"mode": f(self.mode), "success": f(self.test_success).astype(bool), "test_ticks": f(self.test_ticks),
                "test_time": f(self.test_ticks) * self.tick_seconds, "test_best_distance": f(self.test_best_distance),
                "penalty": f(self.penalty).astype(bool), "demos_bought": f(self.demos_bought), "resets_bought": f(self.resets_bought),
                "steps_bought": f(self.steps_bought)}

    def _device_tick(self):
        if self.fused:
            return self._device_tick_fused()
        env, robot = self.env, self.robot
        types = robot.advance_action_types()                                  # int8 [N]
        z = None
        if self.noise == "randn":
            z = self._z.normal_()
        self._prev.copy_(env._state)
        state = self._prev.t()
        action = robot.get_next_action_training(state, None, noise=z, types=types)
        next_state = env.step(action)                                         # null action where the env is not stepping
        robot.process_transition(state, action, next_state, None, types=types)
        env.reset(mask=types, where_equals=2)                                 # the 'reset' envs, straight from the type array
        from . import _lib
        _lib.check(_lib.lib().rtd3_trainer_tally(_lib.ptr(types), _lib.ptr(self.steps_bought), _lib.ptr(self.resets_bought), self.n,
                                                 _lib.stream_ptr(self.device)), "trainer_tally")
        return types

    def _tick_state(self):
        """`rtd3_tick_state` over this trainer's arrays (device pointers; rebuilt per call because the demonstration set and
        the actor input may have been replaced since the last one)."""
        from . import _lib
        env, robot, rb = self.env, self.robot, self.robot.memory
        p = lambda t: None if t is None else t.data_ptr()
        t = _lib.TickStateStruct()
        t.n = self.n
        t.x, t.y, t.goal, t.region, t.state64 = p(env._state[0]), p(env._state[1]), p(robot._goal), p(env._region), p(env._state64)
        t.env_bank = env._bank._struct
        for k in ("num_episodes", "demo_flag", "plan_index", "path_length", "goal_reached", "stuck_flag", "noise_scale", "hist", "hist_count",
                  "hist_head", "type", "update", "any_update", "base", "reward", "reward64", "done"):
            setattr(t, k, p(getattr(robot, "_" + k)))
        t.ax, t.ay = p(robot._action[0]), p(robot._action[1])
        t.prev_x, t.prev_y = p(self._prev[0]), p(self._prev[1])
        t.demo, t.demo_list_start, t.demo_list = p(robot._demo_dev), p(robot._demo_cells), p(robot._demo_list)
        t.num_demo = 0 if robot._demo_dev is None else robot._demo_dev.shape[0]
        t.rp_s, t.rp_a, t.rp_r, t.rp_s2, t.rp_notdone = p(rb.s), p(rb.a), p(rb.r), p(rb.s2), p(rb.notdone)
        t.capacity, t.rp_total = rb.capacity, p(rb._total_dev)
        t.steps_bought, t.resets_bought = p(self.steps_bought), p(self.resets_bought)
        t.philox_seed, t.tick_counter = self.philox_seed, p(self._tick_counter)
        if robot._env_demo is not None:
            d = robot._env_demo
            t.env_demo_pts, t.env_demo_cells, t.env_demo_count, t.env_demo_cap = p(d["sorted"]), p(d["cells"]), p(d["count"]), d["cap"]
        if self.scheduler:
            t.mode, t.demos_bought, t.test_ticks, t.test_best = p(self.mode), p(self.demos_bought), p(self.test_ticks), p(self.test_best_distance)
            t.test_success, t.penalty = p(self.test_success), p(self.penalty)
            t.tick_seconds, t.test_timeout_ticks = self.tick_seconds, self.test_timeout_ticks
        return t

    def _device_tick_fused(self):
        from . import _lib
        from .learner import NET_ACTOR
        env, robot = self.env, self.robot
        if self.n > robot.memory.capacity:
            raise ValueError("more envs than replay rows: raise buffer_size")
        L, sp = _lib.lib(), _lib.stream_ptr(self.device)
        t = self._tick_state()
        _lib.check(L.rtd3_tick_pre(_lib.ctypes.byref(t), sp), "tick_pre")
        z, mode = None, _lib.TICK_NOISE_PHILOX
        if self.noise == "mt19937":
            z, mode = robot.generate_noise(types=robot._type), _lib.TICK_NOISE_GIVEN
        elif self.noise == "randn":
            z, mode = self._z.normal_(), _lib.TICK_NOISE_GIVEN
        residual = robot.td3_agent.forward(NET_ACTOR, robot._base)            # residual_action, robot.py:598-624
        _lib.check(L.rtd3_tick_post(env._handle, _lib.ctypes.byref(t), _lib.ptr(residual), _lib.ptr(z), mode, sp), "tick_post")
        robot.memory._mark_device_advanced()
        return robot._type

    def _multi_tick_ok(self):
        """`rtd3_tick_run_f16` applies: fused ticks, f16 actor forward (2 x H), Philox noise, candidate lists or no demo states."""
        agent, robot = self.robot.td3_agent, self.robot
        # one 128-env tile per CTA: with more tiles than SMs a CTA runs its tiles one after the other (all ticks of one, then of
        # the next) and the three-launch tick, which overlaps them, is faster (65 536 envs: 60 against 36 us per tick)
        one_wave = (self.n + 127) // 128 <= torch.cuda.get_device_properties(self.device).multi_processor_count
        # CTAs of the multi-tick launch drift apart by up to K ticks: everything a launch can push must fit in the ring, otherwise
        # two CTAs could reserve the same slot (rows mixing two transitions) - the three-launch tick serialises and has no such bound
        fits = self.check_interval * self.n <= robot.memory.capacity
        return (self.fused and self.multi_tick_kernel and one_wave and fits and self.noise == "philox" and agent._f16_ok(self.n)
                and (robot._demo_dev is None or robot._demo_cells is not None))

    def _run_multi_tick(self, K):
        from . import _lib
        agent = self.robot.td3_agent
        if self.n > self.robot.memory.capacity:
            raise ValueError("more envs than replay rows: raise buffer_size")
        agent.prepare_forward(self.n)
        t = self._tick_state()
        _lib.check(_lib.lib().rtd3_tick_run_f16(self.env._handle, _lib.ctypes.byref(t), agent.hidden, agent.layers, _lib.ptr(agent.params),
                                                _lib.ptr(agent.params_h), _lib.TICK_NOISE_PHILOX, K, self.ticks, _lib.stream_ptr(self.device)),
                   "tick_run_f16")
        self.robot.memory._mark_device_advanced()
        self._types = self.robot._type

    def run(self, ticks):
        """`ticks` ticks, `check_interval` at a time (the finished-episode counter is read, and a due `td3_update` runs, between
        the blocks exactly where `tick()` would do it).  A block is ONE launch of the multi-tick kernel when `_multi_tick_ok()`,
        else - with `graph=True, fused=True` - one replay of a graph holding `check_interval` fused ticks."""
        K = self.check_interval
        done = 0
        while done < ticks:
            if self._demo_tick_due():
                self.tick()
                done += 1
            elif self._multi_tick_ok() and self.ticks % K == 0 and ticks - done >= K:
                self._run_multi_tick(K)
                self.ticks += K
                done += K
                self.env._state_np = None
                self._maybe_update()
            elif self._use_graph and self.fused and K > 1 and self.ticks % K == 0 and ticks - done >= K:
                self.robot.td3_agent.prepare_forward(self.n)
                self._check_graphs()
                if self._graph_k is None:
                    self.robot.td3_agent._row_scratch(self.robot.td3_agent.batch_size)
                    g = torch.cuda.CUDAGraph()
                    before = _launches()
                    with _capture(g):
                        for _ in range(K):
                            self._types = self._device_tick()
                    self._graph_k, self._graph_k_launches = g, _launches() - before
                    _add_launches(-self._graph_k_launches)
                self._graph_k.replay()
                _add_launches(self._graph_k_launches)
                self.robot.memory._mark_device_advanced()
                self.ticks += K
                done += K
                self.env._state_np = None
                self._maybe_update()
            else:
                self.tick()
                done += 1

    def _maybe_update(self):
        return self.robot.maybe_update_async() if self.async_check else self.robot.maybe_update()

    def _check_graphs(self):
        """A captured tick holds the device pointers of the demonstration set, the env's map configuration (bank and index
        addresses, K, index length) and the choice of forward kernel: drop the graphs when any has changed since the capture
        (`set_demonstration_states`, `process_demonstration`, `set_maps` / `set_map_index`, `precision`)."""
        robot, agent = self.robot, self.robot.td3_agent
        p = lambda t: None if t is None else t.data_ptr()
        # of the operand copies only the one this precision's forward reads (the learner allocates `params_u` at its first
        # tensor-core-mode update: with it in the signature the f16 tick was re-captured - a gc.collect() and 24 launches - right
        # after the first update, inside whatever was being timed)
        fwd = p(agent.params_h) if agent._f16_ok(self.n) else (p(agent.params_u) if agent._tc_ok(self.n) else None)
        ed = robot._env_demo
        sig = (p(robot._demo_dev), p(robot._demo_cells), p(robot._demo_list), agent.precision, fwd,
               None if ed is None else (p(ed["sorted"]), p(ed["cells"]), ed["cap"]), self.env._map_config())
        if sig != getattr(self, "_graph_sig", None):
            self._graph = self._graph_k = None
            self._graph_sig = sig

    def _demo_tick_due(self):
        from .robot import NUM_DEMO
        return self.demonstrations and self.ticks < NUM_DEMO

    def _buy_demonstrations(self):
        """The 'demo' branch of update(dt) for all envs (robot-learning.py:88-92); the tick kernels have already advanced the
        state machine and - with the scheduler - charged the demonstration."""
        states, actions = self.env.get_demonstration()
        self.robot.process_demonstration(states, actions, None)
        self._graph = self._graph_k = None                  # the per-env sets may have been (re)allocated

    def tick(self):
        if self._demo_tick_due():
            types = self._device_tick()
            self._buy_demonstrations()
            self.ticks += 1
            self.env._state_np = None
            if self.ticks % self.check_interval == 0:
                self._maybe_update()
            return types
        if self._use_graph:
            self.robot.td3_agent.prepare_forward(self.n)      # (allocates the operand copies the signature below looks at)
            self._check_graphs()
            if self._graph is None:
                self.robot.td3_agent._row_scratch(self.robot.td3_agent.batch_size)
                g = torch.cuda.CUDAGraph()
                before = _launches()
                with _capture(g):
                    self._types = self._device_tick()
                self._graph, self._graph_launches = g, _launches() - before
                _add_launches(-self._graph_launches)
            self._graph.replay()
            _add_launches(self._graph_launches)
            self.robot.memory._mark_device_advanced()                         # rows were pushed by the replayed kernels
            types = self._types
        else:
            types = self._device_tick()
        self.ticks += 1
        self.env._state_np = None                                             # the kernels moved the state under the host cache
        if self.ticks % self.check_interval == 0:
            self._maybe_update()                                         # robot-learning.py:68 -> robot.py:480-483
        return types


def _capture(graph):
    from . import _lib
    return _lib.capture(graph)


def _launches():
    from . import _lib
    return _lib.launch_count()


def _add_launches(n):
    from . import _lib
    _lib.lib().rtd3_launch_count_add(n)
