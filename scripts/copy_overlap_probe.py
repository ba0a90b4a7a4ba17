"""Does a concurrent pinned H2D copy slow down (a) a cuBLAS bf16 GEMM loop, (b) the min-distance kernel?"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from anomaly_clustering_b200 import ops, pipeline  # noqa: E402

host = torch.empty(482 * 1024 * 1024 // 4, dtype=torch.float32).pin_memory()
dev = torch.empty_like(host, device="cuda")
copy_stream = torch.cuda.Stream()
a = torch.randn(8192, 8192, device="cuda", dtype=torch.bfloat16)
b = torch.randn(8192, 8192, device="cuda", dtype=torch.bfloat16)
n, P, D = 100, 784, 4096
Z = torch.randn(n, P, D, device="cuda") * 0.6
ps = pipeline.patchset_from_Z(Z, "f16")
del Z


def gemm():
    for _ in range(24):
        torch.matmul(a, b)


def mind():
    ops.min_dist_sym(ps.hi, None, ps.n2, 0, ps.hi, None, ps.n2, n, P, "f16")


def t(fn, with_copy):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if with_copy:
        with torch.cuda.stream(copy_stream):
            dev.copy_(host, non_blocking=True)
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


out = torch.empty(n, n * P, dtype=torch.float32, device="cuda")


def mind_full():
    ops.min_dist(ps.hi, None, ps.n2, ps.hi, None, ps.n2, n, P, "f16", out=out)


def mind_half():   # all-pairs kernel on half the queries: same duration class as sym
    ops.min_dist(ps.hi[: 50 * P], None, ps.n2[: 50 * P], ps.hi, None, ps.n2, n, P, "f16", out=out[:, : 50 * P].contiguous())


big = torch.randn(64 * 1024 * 1024, device="cuda")


def elementwise():
    x = big
    for _ in range(40):
        x = x * 1.0001 + 0.5


def report(name, fn):
    t(fn, False)
    print("%-34s alone %.2f ms   with concurrent 482 MB H2D %.2f / %.2f ms" % (name, t(fn, False), t(fn, True), t(fn, True)), flush=True)


report("cuBLAS bf16 8192^3 x24", gemm)
report("torch elementwise x40 (HBM-bound)", elementwise)
report("mindist sym", mind)
report("mindist all-pairs half", mind_half)
