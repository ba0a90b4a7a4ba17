"""GPU bring-up of the tcgen05 min-distance kernel: each configuration runs in its own process so a
trap / deadlock cannot poison the next one.  python scripts/bringup_tc.py"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = [
    # (N_img, P, D, precision)
    (2, 64, 64, "f16"),
    (3, 784, 256, "f16"),
    (3, 100, 1024, "bf16"),
    (3, 784, 512, "f16x3"),
    (5, 784, 4096, "f16"),
]


def child(n, P, D, prec):
    import torch
    from anomaly_clustering_b200 import ops, pipeline

    torch.manual_seed(0)
    base = torch.randn(1, P, D)
    Z = (base + 0.5 * torch.randn(n, P, D)).cuda()
    ps = pipeline.patchset_from_Z(Z, prec)
    dmin = ops.min_dist(ps.hi, ps.lo, ps.n2, ps.hi, ps.lo, ps.n2, n, P, prec)
    torch.cuda.synchronize()
    # exact check from the operands the MMA saw (fp64 on device via torch as a CHECKER only)
    op = ps.hi.double() + (ps.lo.double() if ps.lo is not None else 0)
    op = op.reshape(n, P, D)
    ref = torch.empty(n, n * P, dtype=torch.float64, device="cuda")
    for j in range(n):
        d = torch.cdist(op.reshape(n * P, D), op[j])  # [nP, P]
        ref[j] = d.min(dim=1)[0]
    err = (dmin.double() - ref).abs().max().item()
    mask = torch.ones_like(ref, dtype=torch.bool)
    for j in range(n):
        mask[j, j * P:(j + 1) * P] = False
    err_off = (dmin.double() - ref).abs()[mask].max().item()
    # off-diagonal scale
    print("n=%d P=%d D=%d %s  max|dmin-ref|=%.3e offdiag=%.3e ref-mean=%.3f dmin-mean=%.3f" % (n, P, D, prec, err, err_off, ref.mean().item(), dmin.mean().item()))
    ok = err_off < 2e-2 and err < 0.3
    sys.exit(0 if ok else 3)


if __name__ == "__main__":
    if len(sys.argv) > 1:
        child(int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3]), sys.argv[4])
    fails = 0
    for c in CASES:
        try:
            r = subprocess.run([sys.executable, __file__, *[str(x) for x in c]], capture_output=True, text=True, timeout=120)
            tail = (r.stdout + r.stderr).strip().splitlines()[-3:]
            print("case", c, "rc", r.returncode, "|", " / ".join(tail))
            fails += r.returncode != 0
        except subprocess.TimeoutExpired:
            print("case", c, "TIMEOUT")
            fails += 1
    print("bringup fails:", fails)
