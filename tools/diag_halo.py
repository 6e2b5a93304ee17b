"""2-rank experiment (torchrun): where do the extra microseconds per step of a partitioned run come from?
  A: two INDEPENDENT whole lattices, one per GPU, stepped at the same time (no coupling)
  B: the row-strip pair (halo exchange + waits)"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "spiking-neural-networks_b200"))
import numpy as np, torch, torch.distributed as dist
import bench
from snn_b200 import _capi as K
from snn_b200.backend import CudaLatticeBackend
from snn_b200.dist import StripLattice

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
local = int(os.environ.get("LOCAL_RANK", rank))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
rows = int(sys.argv[1]) if len(sys.argv) > 1 else 3163
cols, iters, reps = 3163, 200, 6
n = rows * cols
f = bench.init_fields(np, n, 0x5EED + rank)
whole = CudaLatticeBackend(K.MODEL_IZH, 0, 0, rows, cols, device=local)
bench.configure(whole, f)
sl = StripLattice(K.MODEL_IZH, rows * world, cols, rank, world, device=local)
bench.configure(sl.be, f)
sl.attach()
for be in (whole, sl.be):
    for _ in range(2):
        be.run_timed(iters)
out = {"A": [], "B": []}
for rep in range(reps):
    for mode, be in (("A", whole), ("B", sl.be)):     # interleaved: thermal / power-cap drift hits both alike
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        ms, nl = be.run_timed(iters)
        out[mode].append(ms * 1e3 / iters)
dist.barrier()
for mode in "AB":
    print(f"[mode {mode} rank {rank}] us per timestep: " + " ".join(f"{t:.1f}" for t in out[mode]), flush=True)
dist.destroy_process_group()
