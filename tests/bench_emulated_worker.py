"""bench.py's own control flow (steady-state leg, collective teardown, end-to-end leg, the JSON line) on a machine
without GPUs: one rank of `bench.py --workload toy` on top of the CUDA emulation of tests/emu, with the handful of
torch.cuda / NCCL calls of bench.py redirected to the host and gloo.  Launched by tests/test_emulated_bench.py
(torchrun for world_size > 1).  Nothing here measures anything: it checks that the benchmark driver itself cannot
stall or crash in the multi-rank orchestration."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "emu", "_pkg"))
sys.path.insert(1, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

torch.cuda.set_device = lambda *args, **kwargs: None
torch.cuda.synchronize = lambda *args, **kwargs: None
_init_process_group, _tensor = dist.init_process_group, torch.tensor
dist.init_process_group = lambda backend, **kwargs: _init_process_group("gloo")
torch.tensor = lambda data, **kwargs: _tensor(data, **{k: v for k, v in kwargs.items() if k != "device"})

import bench  # noqa: E402
from graphvite_b200 import distributed  # noqa: E402


class NoClocks(object):  # nvidia-smi is not here
    def __init__(self, device):
        pass

    def stop(self):
        return {"sm_mhz": 0, "sm_max_mhz": 0, "reasons": []}


def make_solver(cfg, graph, rank, world, local_rank, num_partition=0):
    """bench.make_solver with the exchange moved to host buffers over gloo (emulated device memory is host memory)"""
    import graphvite_b200 as gv
    solver = gv.solver.GraphSolver(cfg["dim"], device_ids=[0], rank=rank, world_size=world)
    if world > 1:
        distributed.attach(solver, None)
    solver.build(graph, gv.optimizer.SGD(cfg["lr"], cfg["weight_decay"]), num_partition=num_partition,
                 num_negative=cfg["num_negative"], batch_size=cfg["batch_size"], episode_size=cfg["episode_size"])
    return solver


bench.ClockSampler = NoClocks
bench.make_solver = make_solver
sys.argv = ["bench.py", "--workload", "toy", "--gpus", os.environ.get("WORLD_SIZE", "1"), "--steps", "4", "--warmup",
            "2", "--no-cpu-baseline", "--watchdog", "0"]
if os.environ.get("GV_BENCH_DUMP"):
    sys.argv += ["--dump-outputs", os.environ["GV_BENCH_DUMP"]]
bench.main()
