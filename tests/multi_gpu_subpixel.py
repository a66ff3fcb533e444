"""torchrun --nproc-per-node 2: the split use_mcc_batch (slab upload + NCCL all-gathers) with subpixel=True must equal
the single-GPU refined table."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
from sea_ice_drift_b200 import synthetic as syn, pmlib
from sea_ice_drift_b200.sharding import use_mcc_batch_split
rank = int(os.environ["RANK"]); local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=3, side=3000, grid=50)
b = np.floor(np.random.default_rng(5).uniform(20, 41, b.size))
split = use_mcc_batch_split(c1, r1, c2, r2, b, img1, img2, 35, 0.0, angles=cfg["angles"], subpixel=True)
single = pmlib.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, angles=cfg["angles"], subpixel=True)
plain = pmlib.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, angles=cfg["angles"])
same = split.tobytes() == single.tobytes() and not np.array_equal(single[:, :2], plain[:, :2], equal_nan=True)
flag = torch.tensor([1 if same else 0], device="cuda")
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0:
    print("subpixel split(%d ranks) == single GPU: %s" % (dist.get_world_size(), bool(flag.item())))
dist.destroy_process_group()
sys.exit(0 if same else 1)
