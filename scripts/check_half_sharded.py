"""torchrun --nproc-per-node N scripts/check_half_sharded.py : the query-sharded path (run_path_sharded) on bf16 and fp16
feature maps against the same path on those maps upcast to fp32.  The 16-bit maps are read natively by the embed
kernels, so w, alpha, X and Dmat must be bit-identical.  Prints one line per dtype ending in OK or MISMATCH."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from anomaly_clustering_b200 import distributed, synth  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
ok = True
n_img, layers, Dp, D = 11, [(768, 28, 28, True), (768, 28, 28, True)], 2048, 4096
lo, hi = distributed.shard_bounds(n_img, world)[rank]
feats, _ = synth.planted_features_device(range(lo, hi), layers, device="cuda")
for dt in (torch.bfloat16, torch.float16):
    f16 = [f.to(dt) for f in feats]
    got = distributed.run_path_sharded(f16, n_img, 3, 1, Dp, D, [1.0, 2.0])
    ref = distributed.run_path_sharded([f.float() for f in f16], n_img, 3, 1, Dp, D, [1.0, 2.0])
    same = [torch.equal(a, b) for a, b in zip(got, ref)]
    good = all(same)
    ok &= good
    if rank == 0:
        print("%s maps, N=%d on %d ranks: a64 / X / Dmat / w bit-identical %s  %s" % (dt, n_img, world, same, "OK" if good else "MISMATCH"),
              flush=True)
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 1)
