"""torchrun --nproc-per-node N scripts/check_sharded.py : the query-sharded multi-GPU path against the single-GPU path on the
same synthetic images; uneven shards included.  Three variants: the default (symmetric-memory transport where it can be set
up), the NCCL collectives (forced in-process through SymmetricBank.disabled_reason) and the all-pairs form."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from anomaly_clustering_b200 import distributed, pipeline, synth  # noqa: E402
from anomaly_clustering_b200.symm_transport import SymmetricBank  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
ok = True
for n_img, layers, Dp, D in ((13, [(96, 12, 12, True), (96, 12, 12, True)], 256, 512),
                             (21, [(768, 28, 28, True), (768, 28, 28, True)], 2048, 4096)):
    bounds = distributed.shard_bounds(n_img, world)
    lo, hi = bounds[rank]
    feats, _ = synth.planted_features_device(range(lo, hi), layers, device="cuda")
    for variant in ("default", "nccl", "all-pairs"):
        saved = SymmetricBank.disabled_reason
        if variant == "nccl":
            SymmetricBank.disabled_reason = "NCCL collectives forced by scripts/check_sharded.py"
        try:
            a64, X, Dm, w = distributed.run_path_sharded(feats, n_img, 3, 1, Dp, D, [1.0, 2.0], symmetric=variant != "all-pairs")
        finally:
            SymmetricBank.disabled_reason = saved
        if rank == 0:
            allf, _ = synth.planted_features_device(range(n_img), layers, device="cuda")
            ref = pipeline.run_path(allf, 3, 1, Dp, D, "unsupervised", [1.0, 2.0])
            e_w = ((w - ref.w[lo:hi]).abs() / ref.w[lo:hi]).max().item()
            e_a = (a64 - ref.alpha64[:, lo:hi]).abs().max().item()
            e_x = ((X - ref.X).norm() / ref.X.norm()).item()
            e_d = ((Dm - ref.Dmat).norm() / ref.Dmat.norm()).item()
            good = e_w < 2e-4 and e_a < 1e-3 and e_x < 1e-4 and e_d < 1e-4
            ok &= good
            print("N=%d images on %d ranks %s  %-9s: w rel %.1e  alpha abs %.1e  X relL2 %.1e  Dmat relL2 %.1e  %s"
                  % (n_img, world, [b - a for a, b in bounds], variant, e_w, e_a, e_x, e_d, "OK" if good else "MISMATCH"), flush=True)
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 1)
