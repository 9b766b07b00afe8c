import os, sys, torch, traceback, collections
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from samble_b200 import models, ops
from samble_b200.config import seg_config
from samble_b200.testing import fill_state_dict_, synthetic_clouds
B, N = 16, 2048
m = models.ShapeNetModel(seg_config(M=(N // 2, N // 4))); m.load_state_dict(fill_state_dict_(m.state_dict(), seed=1, sharpen=4.0)); m = m.eval().cuda()
x, cat = synthetic_clouds(B, N, 2); x, cat = x.cuda(), cat.cuda()
real = ops.transpose12
log = []
def tr(t):
    fr = [f for f in traceback.extract_stack()[:-1] if "samble_b200" in f.filename][-3:]
    log.append((tuple(t.shape), tuple(t.stride()), " <- ".join(f"{f.filename.split('/')[-1]}:{f.lineno}" for f in reversed(fr))))
    return real(t)
with torch.no_grad():
    m(x, cat); models.freeze_boundaries(m)
    ops.transpose12 = tr
    m(x, cat)
for l in log: print(l)
