"""Deviation profile of the whole reference run (tests/test_loop_gpu.py::test_whole_driver_loop_vs_reference): max |state - reference|
per number of completed TD3 updates."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, rtd3_b200 as pkg
g = np.load("tests/golden/loop_golden.npz", allow_pickle=True); e = np.load("tests/golden/env_golden.npz")
torch.manual_seed(0)
loop = pkg.DriverLoop.from_seed(1707366464, maps=(e["speed"], e["angle"]), tick_seconds=float(g["tick_seconds"]))
environment, robot = loop.environment, loop.robot
upd = {"n": 0, "losses": []}
real_update = robot.td3_agent.td3_update
def update_with_recorded_noise(memory):
    z = torch.from_numpy(g["update_noise"][upd["n"] * 100:(upd["n"] + 1) * 100]).cuda()
    upd["losses"].append(real_update(memory, noise=z)); upd["n"] += 1
robot.td3_agent.td3_update = update_with_recorded_noise
demos = {"n": 0}
real_demo = environment.get_demonstration
def demonstration_from_golden():
    real_demo(); k = demos["n"]; demos["n"] += 1
    return g["demo_states"][k], g["demo_actions"][k]
environment.get_demonstration = demonstration_from_golden
dev = {}
for t in range(g["kinds"].shape[0]):
    kind = loop.update()
    k = int(g["kinds"][t])
    if k in (0, 5):
        d = float(np.abs(loop.state - g["states"][t]).max())
        dev[upd["n"]] = max(dev.get(upd["n"], 0.0), d)
        loop.state = g["states"][t].copy(); environment.robot_state = loop.state
print("max |state - reference| by updates done:", {k: round(v, 5) for k, v in sorted(dev.items())})
closs = torch.cat([l[0] for l in upd["losses"]]).cpu().numpy(); aloss = torch.cat([l[1] for l in upd["losses"]]).cpu().numpy()
rc = np.abs(closs / g["critic_losses"] - 1).reshape(-1, 100, 2).max(axis=(1, 2)); ra = np.abs(aloss / g["actor_losses"] - 1).reshape(-1, 50).max(axis=1)
print("max rel critic-loss deviation per update:", np.round(rc, 5).tolist())
print("max rel actor-loss deviation per update:", np.round(ra, 5).tolist())
print("final actor max |dp|:", float(np.abs(robot.td3_agent.flat(0).cpu().numpy() - g["final_actor"]).max()))
