import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from samble_b200 import ops, _lib as L
dev = torch.device("cuda:0")
def t(fn, name):
    for _ in range(3): fn()
    torch.cuda.synchronize(); L.profile(True)
    for _ in range(10): fn()
    torch.cuda.synchronize(); rep = L.profile_report(); L.profile(False)
    print(name, {k: round(v[1] / v[0] * 1e3, 1) for k, v in rep.items()})
B = 16
for (M, N) in [(1024, 2048), (512, 1024)]:
    q = torch.randn(B, M, 128, device=dev); k = torch.randn(B, N, 128, device=dev); v = torch.randn(B, 128, N, device=dev)
    lg = torch.matmul(q, k.transpose(1, 2)) / 11.3
    rm = lg.max(-1)[0]; rs = torch.exp(lg - rm.unsqueeze(-1)).sum(-1)
    t(lambda: ops.cloud_matmul(q, k, row_max=rm, row_sum=rs, logit_div=11.3), f"QK M={M} N={N}")
    p = ops.cloud_matmul(q, k, row_max=rm, row_sum=rs, logit_div=11.3)
    t(lambda: ops.cloud_matmul(p, v), f"PV M={M} N={N}")
