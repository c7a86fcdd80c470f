"""Data-parallel background checkpoint check, run under torchrun with 2 (or more) ranks, one per GPU; the collective comes from
RTD3_DP_COLLECTIVE ("p2p" or "nccl").  argv[1]: a directory every rank can write.

1. A background save, then training (an update and ticks) while the writers run, then the collective `wait()`: fresh objects loaded
   from the directory hold the state at the call on every rank, an update from there equals the original's update after the
   call, and the learner replicas are identical.
2. A second background save into the same directory with rank 1's writer failing: `wait()` raises on every rank, and the directory
   has no manifest (the call removed the first save's)."""
import os
import sys

sys.path[:0] = [os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests")]
import torch
import torch.distributed as dist

import rtd3_b200 as rt
from importlib import import_module
from oracle import env_oracle as eo
from test_checkpoint_gpu import assert_same_state

ck = import_module("residual-td3-robot-navigation_b200.checkpoint")


def main():
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("RTD3_HANG_DUMP_S", "300")), exit=True)
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    path = os.path.join(sys.argv[1], "dp_bg_ckpt")

    def make(seed):
        torch.manual_seed(seed * 100 + rank)
        env = rt.Environment(num_envs=512, seed=1000 * rank + seed, maps=eo.synthetic_maps(0))
        robot = rt.Robot(env._goal.t(), hidden=256, layers=2, seed=10 * rank + seed, buffer_size=1 << 15, process_group=dist.group.WORLD)
        robot.episodes_per_update = 1 << 30                 # updates are run by hand below
        robot.memory.sampler = "philox"
        return rt.BatchedTrainer(env, robot, fused=True, noise="philox")

    def update(tr):
        tr.robot.td3_agent.td3_update(tr.robot.memory)
        torch.cuda.synchronize()
        return tuple(tr.robot.td3_agent.replica_checksum().tolist())

    tr = make(1)
    tr.run(40)
    update(tr)
    sd = tr.state_dict()
    p = rt.save_checkpoint(path, tr, background=True)
    a = update(tr)                                          # training while the writers run
    tr.run(16)
    update(tr)
    assert p.wait() == path
    fresh = make(2)
    rt.load_checkpoint(path, fresh)
    try:
        assert_same_state(fresh.state_dict(), sd)
        state_ok = True
    except AssertionError:
        state_ok = False
    b = update(fresh)
    same = rt.trainer.replicas_identical(tr.robot.td3_agent) and rt.trainer.replicas_identical(fresh.robot.td3_agent)

    real = ck._atomic_save
    if rank == 1:
        def failing(payload, file):
            raise OSError("injected writer failure on rank 1")
        ck._atomic_save = failing
    p2 = rt.save_checkpoint(path, tr, background=True)
    try:
        p2.wait()
        raised = False
    except (OSError, RuntimeError):
        raised = True
    ck._atomic_save = real
    dist.barrier()
    no_manifest = not os.path.exists(os.path.join(path, "manifest.json"))

    ok = state_ok and a == b and same and raised and no_manifest
    flags = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    ok = bool(flags.item())
    print("rank %d: state at the call %s, A %s B %s, replicas identical %s, failure raised %s, no manifest %s"
          % (rank, state_ok, a, b, same, raised, no_manifest), flush=True)
    if rank == 0:
        print("checkpoint background DP%d %s (%s)" % (world, "OK" if ok else "FAIL", tr.robot.td3_agent.dp_collective))
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
