"""torchrun worker: every rank solves its row block twice, once from host arrays (MatCreateMPIAIJWithArrays) and once from device
tensors (MatB200CreateAIJWithDeviceArrays, tensors zeroed right after the constructor), and the two runs must agree bit for bit."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import torch
    import torch.distributed as dist
    from mgpu_worker import build_problem
    rank, size = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    from permon_b200 import api as P
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    P.call("PermonB200SetDevice", local)
    P.initialize()
    dist.init_process_group("nccl", device_id=dev)
    idt = torch.zeros(128, dtype=torch.uint8, device=dev)
    if rank == 0:
        idt.copy_(torch.frombuffer(bytearray(P.get_unique_id()), dtype=torch.uint8))
    dist.broadcast(idt, 0)
    P.comm_init_rank(size, rank, idt.cpu().numpy().tobytes())
    out = {}
    for kind in sys.argv[1].split(","):
        _, loc, _, opts, _ = build_problem(kind, rank, size)
        qtype = "smalxe" if kind.startswith("smalxe") else "mpgp"
        rh = P.solve_problem(loc, qtype, opts)
        rd = P.solve_problem(loc, qtype, opts, device_input="zero")
        same = int(rh.reason == rd.reason and rh.its == rd.its and rh.counts == rd.counts and rh.x.tobytes() == rd.x.tobytes())
        flag = torch.tensor([same], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        out[kind] = dict(identical=bool(flag.item()), its=rh.its, reason=rh.reason)
        dist.barrier()
    if rank == 0:
        print("DEVICE_INPUT_RESULT " + json.dumps(out), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
