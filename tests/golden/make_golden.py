"""Generate golden vectors by running the UNMODIFIED reference (build container only).

    python tests/golden/make_golden.py [env|replay|td3|robot|all]      (and: trace - the configs[0] driver-loop trace)

Imports /root/reference/{environment,robot}.py through oracle/ref_loader.py (import stubs only
for perlin_noise / pyglet / matplotlib, none of which touch hot-path arithmetic) and writes
small .npz fixtures next to this file.  The fixtures travel to the GPU box; the reference does not.
Nothing here is used by the product path.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle.ref_loader import load_reference  # noqa: E402
from oracle.env_oracle import synthetic_maps  # noqa: E402

SEED0 = 1707366464  # configuration.py:26


def make_env():
    env_m, _, constants = load_reference()
    speed, angle = synthetic_maps(0)
    out = {}

    # --- seeding KATs: Environment() then reset() x2 for seeds SEED0 + i  (environment.py:23, 28-56, 130-137)
    n_seed = 64
    goals = np.zeros((n_seed, 2))
    regions = np.zeros((n_seed, 4))
    reset1 = np.zeros((n_seed, 2))
    reset2 = np.zeros((n_seed, 2))
    for i in range(n_seed):
        np.random.seed(SEED0 + i)
        e = env_m.Environment.__new__(env_m.Environment)
        # Environment.__init__ minus set_dynamics (perlin, unpinned, draws nothing from numpy's RNG)
        e.set_init_and_goal()
        goals[i] = e.goal_state
        regions[i] = e.robot_init_region
        reset1[i] = e.reset()
        reset2[i] = e.reset()
    out.update(seed_base=np.int64(SEED0), goals=goals, regions=regions, reset1=reset1, reset2=reset2)

    # --- full constructor KAT of SURVEY 8(c) (uses the stub perlin; RNG stream unaffected)
    np.random.seed(SEED0)
    e = env_m.Environment()
    out.update(kat_region=np.array(e.robot_init_region), kat_goal=np.array(e.goal_state), kat_reset=np.array(e.reset()))

    # --- dynamics / step on the synthetic maps
    e.dynamics_speed = speed
    e.dynamics_angle = angle
    rs = np.random.RandomState(123)
    n = 4096
    states = rs.uniform(0, 98.9999, (n, 2)).astype(np.float32)
    actions = rs.uniform(-7.5, 7.5, (n, 2)).astype(np.float32)
    # edge cases (first rows)
    edge_s = np.array([[0, 0], [98.9999, 98.9999], [0, 98.9999], [50.0, 50.0], [50.0, 50.0], [99 - 2 ** -17, 3.5],
                       [12.999999, 13.0], [0.5, 0.5], [98.5, 98.5], [42.25, 7.75]], dtype=np.float32)
    edge_a = np.array([[-5, -5], [5, 5], [-7, 7], [0, 0], [5, 0], [1, 1],
                       [0.1, -0.1], [-5, -5], [5, 5], [-0.0, 3.0]], dtype=np.float32)
    states[: len(edge_s)] = edge_s
    actions[: len(edge_a)] = edge_a
    nxt64 = np.zeros((n, 2))
    nxt32 = np.zeros((n, 2))
    stp64 = np.zeros((n, 2))
    for i in range(n):
        s64 = states[i].astype(np.float64)
        nxt64[i] = e.dynamics(s64, actions[i].astype(np.float64))     # training-path dtypes (float64 action)
        nxt32[i] = e.dynamics(s64, actions[i])                        # float32 action flow
        e.robot_state = s64
        stp64[i] = e.step(actions[i].astype(np.float64))
    # NaN action: step keeps the state (environment.py:125)
    e.robot_state = np.array([10.0, 20.0])
    nan_kept = np.array(e.step(np.array([np.nan, 1.0])))
    out.update(speed=speed, angle=angle, dyn_states=states, dyn_actions=actions,
               dyn_next_f64act=nxt64, dyn_next_f32act=nxt32, step_next=stp64, nan_kept=nan_kept)

    # --- a 32-step closed-loop rollout of 8 envs (reference runs in float64 state)
    T, m = 32, 8
    acts = rs.uniform(-7.5, 7.5, (T, m, 2)).astype(np.float32)
    traj = np.zeros((T + 1, m, 2))
    for j in range(m):
        e.robot_state = reset1[j].copy()
        traj[0, j] = e.robot_state
        for t in range(T):
            traj[t + 1, j] = e.step(acts[t, j].astype(np.float64))
    out.update(roll_actions=acts, roll_traj=traj)

    # --- environment.compute_reward (environment.py:182-183)
    e.goal_state = goals[0]
    out.update(env_reward=np.float64(e.compute_reward(traj[:, 0])))

    np.savez_compressed(os.path.join(HERE, "env_golden.npz"), **out)
    print("env_golden.npz:", {k: np.asarray(v).shape for k, v in out.items()})


def make_replay():
    _, rob_m, _ = load_reference()
    out = {}
    cases = [(988, 100), (10000, 100), (256, 256), (5000, 256), (10000, 8192 // 8)]
    for ci, (n, B) in enumerate(cases):
        np.random.seed(ci)
        buf = rob_m.ReplayBuffer(10000)
        for k in range(n):
            buf.push(np.array([k, 0.5]), np.array([1.0, k]), float(-k), np.array([k + 1, 0.25]), k % 50 == 49)
        idx_list = []
        rows = None
        for rep in range(3):
            # capture the indices the reference draws: sample() -> np.random.choice(len, B, replace=False)  robot.py:111
            st = np.random.get_state()
            s, a, r, s2, d = buf.sample(B)
            np.random.set_state(st)
            idx = np.random.choice(len(buf), B, replace=False)
            assert (s[:, 0] == idx).all()
            idx_list.append(idx)
            rows = (s, a, r, s2, d)
        out["idx_%d" % ci] = np.stack(idx_list)
        out["case_%d" % ci] = np.array([n, B, ci])
        out["rows_s_%d" % ci], out["rows_a_%d" % ci], out["rows_r_%d" % ci], out["rows_s2_%d" % ci], out["rows_d_%d" % ci] = rows
    # ring wrap-around: capacity 16, push 40 rows (robot.py:79-96)
    buf = rob_m.ReplayBuffer(16)
    for k in range(40):
        buf.push(np.array([k, k]), np.array([k, -k]), float(k), np.array([k, k + 1]), False)
    out["ring_states"] = np.array([t[0] for t in buf.buffer])
    out["ring_position"] = np.int64(buf.position)
    out["under_filled_is_none"] = np.bool_(buf.sample(17) is None)
    np.savez_compressed(os.path.join(HERE, "replay_golden.npz"), **out)
    print("replay_golden.npz written:", len(out), "arrays")


def _flat_params(net):
    import torch
    return torch.cat([p.detach().reshape(-1) for p in net.parameters()]).numpy().copy()


def make_td3():
    """One train_critic, one train_actor, soft_update and a short td3_update of the reference TD3 (robot.py:209-398).

    torch's RNG is never seeded by the reference: weights come from torch.manual_seed(0) here and the
    target-policy noise is captured by wrapping torch.randn_like (the reference code itself is untouched).
    """
    import torch
    _, rob_m, _ = load_reference()
    torch.set_num_threads(1)
    out = {}

    def fill_replay(buf, n, rs, goal):
        for k in range(n):
            s = rs.uniform(0, 98.9999, 2)
            a = rs.uniform(-5, 5, 2)
            s2 = np.clip(s + a, 0, 98.9999)
            r = -np.linalg.norm(s2 - goal)
            buf.push(s, a, r, s2, (k % 50) == 49)

    goal = np.array([86.43404857, 24.75898687])
    rs = np.random.RandomState(7)
    buf = rob_m.ReplayBuffer(10000)
    fill_replay(buf, 2000, rs, goal)
    out["rep_s"] = np.array([t[0] for t in buf.buffer])
    out["rep_a"] = np.array([t[1] for t in buf.buffer])
    out["rep_r"] = np.array([t[2] for t in buf.buffer])
    out["rep_s2"] = np.array([t[3] for t in buf.buffer])
    out["rep_d"] = np.array([t[4] for t in buf.buffer])

    torch.manual_seed(0)
    agent = rob_m.TD3(rob_m.Residual_Actor_Network(), rob_m.Residual_Critic_Network(), rob_m.Residual_Critic_Network())
    # biases are zero at init; perturb them so bias handling is exercised (weights are inputs to both sides)
    with torch.no_grad():
        for net in (agent.actor_network, agent.critic_network_1, agent.critic_network_2):
            for p in net.parameters():
                if p.dim() == 1:
                    p.add_(0.01 * torch.randn_like(p))
        # targets differ from the online nets (as they do after the first Polyak step)
        for net in (agent.target_actor, agent.target_critic_network_1, agent.target_critic_network_2):
            for p in net.parameters():
                p.add_(0.003 * torch.randn_like(p))
    nets = dict(actor=agent.actor_network, critic1=agent.critic_network_1, critic2=agent.critic_network_2,
                t_actor=agent.target_actor, t_critic1=agent.target_critic_network_1, t_critic2=agent.target_critic_network_2)
    for k, net in nets.items():
        out["w0_" + k] = _flat_params(net)

    noises = []
    real_randn_like = torch.randn_like

    def capturing_randn_like(t, *a, **kw):
        z = real_randn_like(t, *a, **kw)
        noises.append(z.numpy().copy())
        return z

    idxs = []
    real_choice = np.random.choice

    def capturing_choice(*a, **kw):
        r = real_choice(*a, **kw)
        idxs.append(np.array(r))
        return r

    torch.randn_like = capturing_randn_like
    np.random.choice = capturing_choice
    try:
        np.random.seed(0)
        torch.manual_seed(1)
        # ---- one critic step (robot.py:312-366)
        l1, l2 = agent.train_critic(buf)
        out["critic_losses"] = np.array([l1, l2])
        for k, net in nets.items():
            out["w1_" + k] = _flat_params(net)
        s = torch.FloatTensor(out["rep_s"][idxs[0]])
        a = torch.FloatTensor(out["rep_a"][idxs[0]])
        with torch.no_grad():
            out["q1_after_critic"] = agent.critic_network_1(s, a).numpy().copy()
            out["q2_after_critic"] = agent.critic_network_2(s, a).numpy().copy()
        # ---- one actor step (robot.py:369-398) then the three soft updates (robot.py:283-285)
        la = agent.train_actor(buf)
        out["actor_loss"] = np.float64(la)
        agent.soft_update(agent.target_actor, agent.actor_network, agent.tau)
        agent.soft_update(agent.target_critic_network_1, agent.critic_network_1, agent.tau)
        agent.soft_update(agent.target_critic_network_2, agent.critic_network_2, agent.tau)
        for k, net in nets.items():
            out["w2_" + k] = _flat_params(net)
        out["idx_critic"] = idxs[0]
        out["idx_actor"] = idxs[1]
        out["noise_critic"] = noises[0]
        # ---- a short full td3_update: 6 epochs (3 actor steps), continuing from the state above
        del idxs[:], noises[:]
        agent.num_epochs = 6
        c_losses, a_losses = [], []
        real_tc, real_ta = agent.train_critic, agent.train_actor

        def tc(rb):
            r = real_tc(rb)
            c_losses.append(r)
            return r

        def ta(rb):
            r = real_ta(rb)
            a_losses.append(r)
            return r

        agent.train_critic, agent.train_actor = tc, ta
        agent.td3_update(buf)
        out["upd_idx"] = np.stack(idxs)            # order: c,a,c,c,a,c,c,a,c  (epochs 0..5, actor on even)
        out["upd_noise"] = np.stack(noises)        # 6 x [B,2]
        out["upd_critic_losses"] = np.array(c_losses)
        out["upd_actor_losses"] = np.array(a_losses)
        for k, net in nets.items():
            out["w3_" + k] = _flat_params(net)
    finally:
        torch.randn_like = real_randn_like
        np.random.choice = real_choice
    np.savez_compressed(os.path.join(HERE, "td3_golden.npz"), **out)
    print("td3_golden.npz written; critic losses", out["critic_losses"], "actor loss", out["actor_loss"])


def make_robot():
    """Per-step hooks of Robot (robot.py:443-675, 727-762) on a deterministic trace."""
    import torch
    env_m, rob_m, constants = load_reference()
    torch.set_num_threads(1)
    speed, angle = synthetic_maps(0)
    out = {}
    np.random.seed(SEED0)
    e = env_m.Environment()
    e.dynamics_speed, e.dynamics_angle = speed, angle
    state = e.reset()
    torch.manual_seed(0)
    robot = rob_m.Robot(e.goal_state)
    out["goal"] = np.array(e.goal_state)
    out["actor_w"] = _flat_params(robot.td3_agent.actor_network)

    # ---- act: get_next_action_training / testing  (robot.py:541-642)
    rs = np.random.RandomState(5)
    S = rs.uniform(0, 98.9999, (64, 2))
    robot.current_noise_scale = 0.75
    np.random.seed(99)
    out["act_states"] = S
    out["act_train"] = np.array([robot.get_next_action_training(s, 100.0) for s in S])
    out["act_test"] = np.array([robot.get_next_action_testing(s) for s in S])
    with torch.no_grad():
        out["act_residual"] = robot.td3_agent.actor_network(torch.FloatTensor(S - e.goal_state)).numpy().copy()
    robot.current_noise_scale = 1

    # ---- reward + stuck + done on a synthetic trace with a demo set  (robot.py:645-675, 727-762, 509-538)
    demo = rs.uniform(20, 80, (500, 2))
    robot.demonstration_states = list(demo)
    robot.demo_flag = True
    robot.path_length = 12
    T = 40
    trace_s = np.zeros((T, 2))
    trace_s2 = np.zeros((T, 2))
    trace_a = rs.uniform(-5, 5, (T, 2))
    cur = np.array([30.0, 30.0])
    for t in range(T):
        trace_s[t] = cur
        step = trace_a[t] * (0.05 if 8 <= t < 20 else 1.0)    # a slow stretch -> stuck detection fires
        nxt = np.clip(cur + step, 0, 98.9999)
        if t == 30:
            nxt = e.goal_state + np.array([3.0, -3.9])        # inside the goal radius
        trace_s2[t] = nxt
        cur = nxt
    rew, done, stuck, reached, plan = [], [], [], [], []
    robot.memory = rob_m.ReplayBuffer(10000)
    robot.plan_index = 0
    for t in range(T):
        robot.process_transition(trace_s[t], trace_a[t], trace_s2[t], 100.0)
        row = robot.memory.buffer[-1]
        rew.append(row[2]); done.append(row[4]); stuck.append(robot.stuck_flag); reached.append(robot.goal_reached)
        plan.append(robot.plan_index)
        # the driver's episode logic (robot.py:480-487) without the td3_update call
        if robot.plan_index == robot.path_length - 1 or robot.goal_reached or robot.stuck_flag:
            robot.plan_index = 0; robot.goal_reached = False; robot.stuck_flag = False
        else:
            robot.plan_index += 1
    out.update(demo_states=demo, trace_s=trace_s, trace_a=trace_a, trace_s2=trace_s2, trace_reward=np.array(rew),
               trace_done=np.array(done), trace_stuck=np.array(stuck), trace_reached=np.array(reached),
               trace_plan=np.array(plan), trace_path_length=np.int64(12))

    # ---- get_next_action_type state machine (robot.py:443-506); td3_update replaced by a counter
    torch.manual_seed(0)
    robot = rob_m.Robot(e.goal_state)
    calls = []
    robot.td3_agent.td3_update = lambda mem: calls.append(1)
    types, eps, noise, plens = [], [], [], []
    for t in range(400):
        if t in (200, 300):
            robot.stuck_flag = True
        if t == 250:
            robot.goal_reached = True
        ty = robot.get_next_action_type(np.zeros(2), 100.0)
        types.append({"step": 0, "demo": 1, "reset": 2}[ty])
        eps.append(robot.num_episodes); noise.append(robot.current_noise_scale); plens.append(robot.path_length)
    out.update(sm_types=np.array(types), sm_episodes=np.array(eps), sm_noise=np.array(noise), sm_path_len=np.array(plens),
               sm_updates=np.int64(len(calls)))
    np.savez_compressed(os.path.join(HERE, "robot_golden.npz"), **out)
    print("robot_golden.npz written")


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    if what in ("env", "all"):
        make_env()
    if what in ("replay", "all"):
        make_replay()
    if what in ("td3", "all"):
        make_td3()
    if what in ("robot", "all"):
        make_robot()


def make_trace():
    """configs[0]: the reference's own driver loop (robot-learning.py:66-101, training branch, without pyglet) on one env:
    seeded start/goal, three demonstrations, the first episodes and the first TD3 update.  The wall-clock money term is
    replaced by zero so that the run is deterministic.  Demonstrations, torch-side randomness (initial weights, target
    noise) and every per-tick observable are recorded."""
    import torch
    env_m, rob_m, constants = load_reference()
    torch.set_num_threads(1)
    speed, angle = synthetic_maps(0)
    np.random.seed(SEED0)
    torch.manual_seed(0)
    environment = env_m.Environment()
    environment.dynamics_speed, environment.dynamics_angle = speed, angle
    state = environment.reset()
    robot = rob_m.Robot(environment.goal_state)
    out = {"goal": np.array(environment.goal_state), "region": np.array(environment.robot_init_region), "state0": np.array(state)}
    for k, net in (("actor", robot.td3_agent.actor_network), ("critic1", robot.td3_agent.critic_network_1), ("critic2", robot.td3_agent.critic_network_2)):
        out["w_" + k] = _flat_params(net)
    noises = []
    real_randn_like = torch.randn_like
    def capturing_randn_like(t, *a, **kw):
        z = real_randn_like(t, *a, **kw)
        noises.append(z.numpy().copy())
        return z
    torch.randn_like = capturing_randn_like
    losses = []
    real_tc, real_ta = robot.td3_agent.train_critic, robot.td3_agent.train_actor
    robot.td3_agent.train_critic = lambda rb: (lambda r: (losses.append(("c",) + r), r)[1])(real_tc(rb))
    robot.td3_agent.train_actor = lambda rb: (lambda r: (losses.append(("a", r)), r)[1])(real_ta(rb))
    types, states, actions, rewards, dones, demos_s, demos_a = [], [], [], [], [], [], []
    demos_bought = resets_bought = steps_bought = 0
    try:
        for tick in range(130):
            money = constants.STARTING_MONEY - (demos_bought * constants.COST_PER_DEMO + resets_bought * constants.COST_PER_RESET +
                                                steps_bought * constants.COST_PER_STEP)
            action_type = robot.get_next_action_type(state, money)
            types.append({"step": 0, "demo": 1, "reset": 2}[action_type])
            act = np.zeros(2)
            if action_type == "reset":
                state = environment.reset()
                resets_bought += 1
            elif action_type == "demo":
                ds, da = environment.get_demonstration()
                demos_s.append(np.array(ds)); demos_a.append(np.array(da))
                robot.process_demonstration(ds, da, money)
                demos_bought += 1
            else:
                act = robot.get_next_action_training(state, money)
                next_state = environment.step(act)
                robot.process_transition(state, act, next_state, money)
                row = robot.memory.buffer[(robot.memory.position - 1) % robot.memory.capacity]
                rewards.append(row[2]); dones.append(row[4])
                state = next_state
                steps_bought += 1
            states.append(np.array(state)); actions.append(np.array(act))
    finally:
        torch.randn_like = real_randn_like
    out.update(types=np.array(types), states=np.array(states), actions=np.array(actions), step_rewards=np.array(rewards),
               step_dones=np.array(dones), demo_states=np.array(demos_s), demo_actions=np.array(demos_a),
               update_noise=np.array(noises, dtype=np.float32), n_updates=np.int64(len(noises) // 100),
               critic_losses=np.array([l[1:] for l in losses if l[0] == "c"]), actor_losses=np.array([l[1] for l in losses if l[0] == "a"]),
               replay_len=np.int64(len(robot.memory)), final_uniform=np.float64(np.random.uniform()))
    np.savez_compressed(os.path.join(HERE, "trace_golden.npz"), **out)
    print("trace_golden.npz: types", np.bincount(types), "updates", out["n_updates"], "replay", out["replay_len"])


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "trace":
    make_trace()


def make_loop():
    """configs[0], the WHOLE run of the reference's driver (robot-learning.py:19-117 without pyglet): training until the money is
    gone (three demonstrations, episodes with their TD3 updates, purchases refused once they are not affordable), the switch to
    testing, the test phase until success or time-out.  The wall-clock money term is charged as 0.1 s per update() call (the
    interval the script schedules update at) and the test time-out is counted in the same ticks - the only changes to the script's
    logic, made so that the run is deterministic (trainer.DriverLoop restates exactly this)."""
    import torch
    env_m, rob_m, constants = load_reference()
    torch.set_num_threads(1)
    speed, angle = synthetic_maps(0)
    np.random.seed(SEED0)
    torch.manual_seed(0)
    environment = env_m.Environment()
    environment.dynamics_speed, environment.dynamics_angle = speed, angle
    state = environment.reset()
    robot = rob_m.Robot(environment.goal_state)
    noises = []
    real_randn_like = torch.randn_like
    def capturing_randn_like(t, *a, **kw):
        z = real_randn_like(t, *a, **kw)
        noises.append(z.numpy().copy())
        return z
    torch.randn_like = capturing_randn_like
    losses = []
    real_tc, real_ta = robot.td3_agent.train_critic, robot.td3_agent.train_actor
    robot.td3_agent.train_critic = lambda rb: (lambda r: (losses.append(("c",) + r), r)[1])(real_tc(rb))
    robot.td3_agent.train_actor = lambda rb: (lambda r: (losses.append(("a", r)), r)[1])(real_ta(rb))
    TICK_SECONDS = 0.1
    timeout_ticks = int(round(constants.TEST_TIMEOUT / TICK_SECONDS))
    mode, ticks = "training", 0
    demos_bought = resets_bought = steps_bought = 0
    test_ticks, test_best, penalty, success, finished = 0, np.inf, False, False, False
    kinds, states, actions, moneys, demos_s, demos_a, step_rewards, step_dones = [], [], [], [], [], [], [], []
    code = {"step": 0, "demo": 1, "reset": 2, "switch": 3, "skip": 4, "test": 5}

    def money_now():
        spent = (demos_bought * constants.COST_PER_DEMO + resets_bought * constants.COST_PER_RESET + steps_bought * constants.COST_PER_STEP
                 + (ticks * TICK_SECONDS) * constants.COST_PER_CPU_SECOND)
        return constants.STARTING_MONEY - spent
    try:
        while not finished:
            act = np.zeros(2)
            if mode == "training":
                money = money_now()
                action_type = robot.get_next_action_type(state, money)
                money = money_now()
                ticks += 1
                moneys.append(money)
                kind = action_type
                if money < 0:
                    penalty = money < -1.0
                    state = environment.reset()
                    mode = "testing"
                    kind = "switch"
                elif action_type == "reset":
                    if money >= constants.COST_PER_RESET:
                        state = environment.reset()
                        resets_bought += 1
                    else:
                        kind = "skip"
                elif action_type == "demo":
                    if money >= constants.COST_PER_DEMO:
                        ds, da = environment.get_demonstration()
                        demos_s.append(np.array(ds)); demos_a.append(np.array(da))
                        robot.process_demonstration(ds, da, money)
                        demos_bought += 1
                    else:
                        kind = "skip"
                else:
                    if money >= constants.COST_PER_STEP:
                        act = robot.get_next_action_training(state, money)
                        next_state = environment.step(act)
                        robot.process_transition(state, act, next_state, money)
                        row = robot.memory.buffer[(robot.memory.position - 1) % robot.memory.capacity]
                        step_rewards.append(row[2]); step_dones.append(row[4])
                        state = next_state
                        steps_bought += 1
                    else:
                        kind = "skip"
            else:
                act = robot.get_next_action_testing(state)
                next_state = environment.step(act)
                distance = np.linalg.norm(next_state - environment.goal_state)
                state = next_state
                test_ticks += 1
                moneys.append(np.nan)
                kind = "test"
                if distance <= constants.TEST_DISTANCE_THRESHOLD:
                    success = finished = True
                if distance < test_best:
                    test_best = distance
                if test_ticks >= timeout_ticks:
                    finished = True
            kinds.append(code[kind]); states.append(np.array(state, dtype=np.float64)); actions.append(np.array(act, dtype=np.float64))
    finally:
        torch.randn_like = real_randn_like
    out = {"goal": np.array(environment.goal_state), "region": np.array(environment.robot_init_region),
           "kinds": np.array(kinds, dtype=np.int8), "states": np.array(states), "actions": np.array(actions), "money": np.array(moneys),
           "step_rewards": np.array(step_rewards, dtype=np.float64), "step_dones": np.array(step_dones),
           "demo_states": np.array(demos_s), "demo_actions": np.array(demos_a),
           "update_noise": np.array(noises, dtype=np.float32), "n_updates": np.int64(len(noises) // 100),
           "critic_losses": np.array([l[1:] for l in losses if l[0] == "c"]), "actor_losses": np.array([l[1] for l in losses if l[0] == "a"]),
           "demos_bought": np.int64(demos_bought), "resets_bought": np.int64(resets_bought), "steps_bought": np.int64(steps_bought),
           "training_ticks": np.int64(ticks), "test_ticks": np.int64(test_ticks), "test_best_distance": np.float64(test_best),
           "success": np.bool_(success), "penalty": np.bool_(penalty), "tick_seconds": np.float64(TICK_SECONDS),
           "final_actor": _flat_params(robot.td3_agent.actor_network), "replay_len": np.int64(len(robot.memory)),
           "final_uniform": np.float64(np.random.uniform())}
    np.savez_compressed(os.path.join(HERE, "loop_golden.npz"), **out)
    print("loop_golden.npz: kinds", np.bincount(kinds), "training ticks", ticks, "test ticks", test_ticks, "success", success,
          "best", test_best, "updates", out["n_updates"], "bought", demos_bought, resets_bought, steps_bought)


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "loop":
    make_loop()


def make_demo():
    """Demonstrations (SURVEY.md 8 f-1 / f-2): the reference's CEM planner (environment.py:140-179) with its random draws recorded
    (np.random.choice / np.random.normal are wrapped to log what they return - the reference itself is untouched), and
    augment_demonstration_data (robot.py:771-823) on the planner's output."""
    import torch
    env_m, rob_m, constants = load_reference()
    speed, angle = synthetic_maps(0)
    out = {}
    for k, seed in enumerate((SEED0, 77)):
        np.random.seed(seed)
        e = env_m.Environment()
        e.dynamics_speed, e.dynamics_angle = speed, angle
        e.reset()
        choices, normals, locs, scales = [], [], [], []
        real_choice, real_normal = np.random.choice, np.random.normal
        def rec_choice(*a, **kw):
            v = real_choice(*a, **kw)
            choices.append(np.array(v))
            return v
        def rec_normal(loc=0.0, scale=1.0, size=None):
            v = real_normal(loc, scale, size)
            normals.append(np.array(v)); locs.append(np.array(loc)); scales.append(np.array(scale))
            return v
        np.random.choice, np.random.normal = rec_choice, rec_normal
        try:
            ds, da = e.get_demonstration()
        finally:
            np.random.choice, np.random.normal = real_choice, real_normal
        P, T = constants.DEMOS_CEM_NUM_PATHS, constants.DEMOS_CEM_PATH_LENGTH
        ch = np.array(choices).reshape(P, T, 2)
        nm = np.array(normals).reshape(3, P, T, 2)
        out.update({"seed_%d" % k: np.int64(seed), "goal_%d" % k: np.array(e.goal_state), "region_%d" % k: np.array(e.robot_init_region),
                    "start_%d" % k: np.array(ds[0], dtype=np.float64), "it0_actions_%d" % k: ch[:4].astype(np.float32),
                    "it1_draws_%d" % k: nm[0, :2], "it1_mean_%d" % k: np.array(locs[:T], dtype=np.float32),
                    "it1_std_%d" % k: np.array(scales[:T], dtype=np.float32),
                    "it3_mean_%d" % k: np.array(locs[2 * P * T:2 * P * T + T], dtype=np.float32),
                    "demo_states_%d" % k: np.array(ds), "demo_actions_%d" % k: np.array(da),
                    "uniform_after_plan_%d" % k: np.float64(np.random.uniform())})
        # augmentation on this demonstration, from a fresh seed
        torch.manual_seed(0)
        robot = rob_m.Robot(e.goal_state)
        np.random.seed(seed + 1)
        robot.augment_demonstration_data(ds, da)
        out.update({"aug_states_%d" % k: np.array([np.asarray(s, dtype=np.float64) for s in robot.demonstration_states]),
                    "uniform_after_aug_%d" % k: np.float64(np.random.uniform())})
        # process_demonstration rows (demo_flag False, as at the reference's call sites)
        robot2 = rob_m.Robot(e.goal_state)
        np.random.seed(seed + 2)
        robot2.process_demonstration(ds, da, 100.0)
        rows = robot2.memory.buffer
        out.update({"rows_reward_%d" % k: np.array([r[2] for r in rows], dtype=np.float64), "rows_done_%d" % k: np.array([r[4] for r in rows]),
                    "rows_state_%d" % k: np.array([r[0] for r in rows]), "n_demo_states_%d" % k: np.int64(len(robot2.demonstration_states))})
    np.savez_compressed(os.path.join(HERE, "demo_golden.npz"), **out)
    print("demo_golden.npz written:", {k: v.shape for k, v in out.items() if hasattr(v, "shape") and v.ndim})


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "demo":
    make_demo()


def make_adam():
    """torch.optim.Adam (the reference's optimiser, robot.py:237-239) on CPU: five steps on 100003 parameters from
    torch.manual_seed(0), recorded on an x86 CPU with torch's AVX-512 kernels (the operation order oracle/td3_oracle.py adam_step
    restates).  The step is elementwise, so a seeded sample of 2048 elements is stored: inputs, exp_avg, exp_avg_sq and parameters
    after every step."""
    import torch
    torch.manual_seed(0)
    n, steps = 100003, 5
    p0 = torch.randn(n)
    par = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([par], lr=1e-3)
    grads, m, v, p = [], [], [], []
    for _ in range(steps):
        g = (torch.randn(n) * 0.05 * torch.rand(n)).numpy().astype(np.float32)
        par.grad = torch.from_numpy(g.copy())
        opt.step()
        grads.append(g)
        m.append(opt.state[par]["exp_avg"].numpy().copy())
        v.append(opt.state[par]["exp_avg_sq"].numpy().copy())
        p.append(par.detach().numpy().copy())
    idx = np.sort(np.random.RandomState(0).choice(n, 2048, replace=False))
    out = {"cpu_capability": np.array(torch.backends.cpu.get_cpu_capability()), "p0": p0.numpy()[idx],
           "grad": np.stack(grads)[:, idx], "exp_avg": np.stack(m)[:, idx], "exp_avg_sq": np.stack(v)[:, idx], "param": np.stack(p)[:, idx]}
    np.savez_compressed(os.path.join(HERE, "adam_golden.npz"), **out)
    print("adam_golden.npz written:", {k: v.shape for k, v in out.items()})


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "adam":
    make_adam()
