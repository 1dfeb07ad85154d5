import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from coevonet_b200 import layout, ops
pitch = layout.fc_pitch(10)
theta = torch.randn(pitch, device="cuda") * 0.05
P = 1024
fit = torch.randn(P, dtype=torch.float64, device="cuda")
def t(fn, n=10):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3
out = torch.empty((P, pitch), device="cuda")
print("K5 perturb us:", t(lambda: ops.es_perturb(theta, 10, 0.05, 1, "agent_0", 0, 0, P, out=out)))
print("K6 regen   us:", t(lambda: ops.es_update(fit, 10, 0.05, 0.1, P, 1, "agent_0", 0, 0)))
print("K6 members us:", t(lambda: ops.es_update_members(fit, out, theta, 10, 0.05, 0.1, P)))
