"""Data-parallel checkpoint check, run under torchrun with 2 (or more) ranks, one per GPU; the collective comes from
RTD3_DP_COLLECTIVE ("p2p" or "nccl").  argv[1]: a directory both ranks can write.

Save a trainer; update the original (checksum A); load into fresh objects and update (B); then, in the same process, roll the live
objects back to the checkpoint and update again (C).  Pass: A == B == C and the replicas are identical.  C catches a restored
peer-memory step counter: receive areas still stamped with later steps would be read as fresh gradients."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

import rtd3_b200 as rt
from oracle import env_oracle as eo


def main():
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("RTD3_HANG_DUMP_S", "300")), exit=True)
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    path = os.path.join(sys.argv[1], "dp_ckpt")

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
    update(tr)                                              # the peer-memory step counter is past zero at the save
    rt.save_checkpoint(path, tr)
    a = update(tr)
    update(tr)                                              # the live areas now hold later steps than the checkpoint's
    fresh = make(2)
    rt.load_checkpoint(path, fresh)
    b = update(fresh)
    rt.load_checkpoint(path, tr)
    c = update(tr)
    same = rt.trainer.replicas_identical(tr.robot.td3_agent) and rt.trainer.replicas_identical(fresh.robot.td3_agent)
    ok = a == b == c and same
    flags = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    ok = bool(flags.item())
    if rank == 0:
        print("checkpoint DP%d %s (%s): A %s B %s C %s replicas identical %s"
              % (world, "OK" if ok else "FAIL", tr.robot.td3_agent.dp_collective, a, b, c, same))
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
