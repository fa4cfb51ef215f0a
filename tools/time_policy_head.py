"""Times drq_policy_head_fwd_bf16 (warm, back to back, CUDA events) against the launches it replaced: the
Linear(hidden, A) as a tensor-core GEMM tile plus two drq_actor_sample launches.  M = 512 rows, A = 6, H = 1024."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from drqv2_b200 import _lib  # noqa: E402
from drqv2_b200._bf16 import TB, PolicySample, gemm  # noqa: E402
from drqv2_b200._lib import GEMM_KK, TEPI_F32  # noqa: E402

dev = torch.device("cuda")
def cur():
    return torch.cuda.current_stream().cuda_stream          # the capture stream inside torch.cuda.graph


M, A, H, B = 512, 6, 1024, 256
g = torch.Generator(device="cuda").manual_seed(0)
p2 = TB(M, H, dev); p2.buf.copy_((torch.rand(p2.buf.numel(), device=dev, generator=g) - 0.3).clamp_min(0).to(torch.bfloat16))
w4 = (torch.rand(A, H, device=dev, generator=g) - 0.5) * 0.1
b4 = torch.zeros(A, device=dev)
w4b = TB(A, H, dev, rblk=64); w4b.load(w4)
mu_pre = torch.zeros(M, A, device=dev)
std = torch.tensor([0.4], device=dev)
ticket = torch.zeros(1 + 4096, dtype=torch.int32, device=dev)
eps = torch.randn(B, A, device=dev, generator=g)
out1, out2, mu = torch.zeros(B, A), torch.zeros(B, A), torch.zeros(B, A)
out1, out2, mu = out1.to(dev), out2.to(dev), mu.to(dev)
metrics = torch.zeros(2, device=dev)
jobs = (PolicySample * 2)(PolicySample(256, B, eps.data_ptr(), out1.data_ptr(), A, None, None, None, 0, 0, 0),
                          PolicySample(0, B, eps.data_ptr(), out2.data_ptr(), A, mu.data_ptr(), metrics.data_ptr(), None, 0, 0, 0))


def fused(nj):
    _lib.call("drq_policy_head_fwd_bf16", p2.ptr(), p2.units, w4.data_ptr(), b4.data_ptr(), mu_pre.data_ptr(), M, H, A, jobs, nj,
              std.data_ptr(), 0.3, ticket.data_ptr(), cur())


def unfused():
    gemm(p2.ptr(), p2.units, w4b.ptr(), w4b.units, GEMM_KK, mu_pre.data_ptr(), A, M, A, H, TEPI_F32, bias=b4.data_ptr())
    _lib.call("drq_actor_sample", mu_pre.data_ptr() + 4 * 256 * A, eps.data_ptr(), std.data_ptr(), 0.3, out1.data_ptr(), A, None, None, B, A, cur())
    _lib.call("drq_actor_sample", mu_pre.data_ptr(), eps.data_ptr(), std.data_ptr(), 0.3, out2.data_ptr(), A, mu.data_ptr(), metrics.data_ptr(), B, A, cur())


def timeit(fn, n=200):
    for _ in range(10):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(20):
            fn()
    graph.replay()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n // 20):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


print("policy head fused, 2 sample jobs : %.2f us" % timeit(lambda: fused(2)))
print("policy head fused, 0 sample jobs : %.2f us" % timeit(lambda: fused(0)))
print("gemm tile + 2 sample launches    : %.2f us" % timeit(unfused))
