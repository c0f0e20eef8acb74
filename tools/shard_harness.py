"""What the sharded-handle tools share: the torchrun demos (one process per GPU, Ranks) and the single-process benches
(gpu_info, pool_stats, timed)."""
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch
import torch.distributed as dist

from multilinear_b200 import api as ml
from multilinear_b200 import load


class Ranks:
    """this torchrun process: its rank, its GPU and (world > 1) the NCCL process group, which only all-gathers the IPC records
    and reduces the results; the data path of the handles is peer stores + device flags"""

    def __init__(self):
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.rank = int(os.environ.get("RANK", 0))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(self.local)
        ml.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def connect(self, sh):
        """the handle's arenas connected to every other process's (to its own at world 1)"""
        if self.world > 1:
            sh.connect_over(dist, self.dev)
        else:
            sh.connect(sh.export())
        return sh

    def barrier(self):
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()

    def timed(self, sh, fn, reps):
        """one warm-up call, then reps calls between CUDA events on the handle's stream, every rank entering together; returns
        (ms per call, the maximum over the ranks; the last call's result)"""
        stream = torch.cuda.ExternalStream(sh.stream(0), device=self.dev)
        self.barrier()
        fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            out = fn()
        e1.record(stream)
        self.barrier()
        ms = e0.elapsed_time(e1) / reps
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms, out

    def agree(self, data):
        """whether every rank holds rank 0's bytes"""
        if self.world == 1:
            return True
        mine = torch.tensor(list(data), dtype=torch.uint8, device=self.dev)
        d0 = mine.clone()
        dist.broadcast(d0, 0)
        flag = torch.tensor([int(torch.equal(mine, d0))], device=self.dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        return bool(int(flag[0]))

    def close(self, sh):
        """free the handle once every rank is done with the peers' arenas, then leave the process group"""
        self.barrier()
        sh.free()
        if self.world > 1:
            dist.barrier()
            dist.destroy_process_group()


def gpu_info():
    """name, power limit and clocks of every GPU, read in the same run as the numbers they qualify"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout
        return [l.strip() for l in out.splitlines() if l.strip()]
    except Exception as e:  # noqa: BLE001
        return ["nvidia-smi unavailable: %s" % e]


def pool_stats(dev):
    """(reserved, used) bytes of the stream-ordered pool on device dev"""
    ml.set_device(dev)
    r, u = C.c_uint64(), C.c_uint64()
    ml.check(load().ml_pool_stats(C.byref(r), C.byref(u)))
    return r.value, u.value


def timed(streams, fn):
    """fn() under CUDA events on every (device, stream); returns (result, max ms over the streams)"""
    evs = []
    for dev, s in streams:
        with torch.cuda.device(dev):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s)
            evs.append((dev, s, e0, e1))
    out = fn()
    for dev, s, e0, e1 in evs:
        with torch.cuda.device(dev):
            e1.record(s)
    for dev, _, _, _ in evs:
        torch.cuda.synchronize(dev)
    return out, max(e0.elapsed_time(e1) for _, _, e0, e1 in evs)
