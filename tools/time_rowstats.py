import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from samble_b200 import ops
B, N, D = 16, 2048, 128
qkv = torch.randn(B, N, 3 * D, device="cuda")
q, k = qkv[..., :D], qkv[..., D:2 * D]
k_tok = torch.randn(4, D, device="cuda")
for fast in (False, True):
    ops._DS_FAST = fast
    ks = ops.split_operand(k) if fast else None
    for _ in range(3):
        ops.ds_row_stats(q, k, k_tok, k_split=ks)
    torch.cuda.synchronize()
print("done")
