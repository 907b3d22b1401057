import sys
sys.path.insert(0, "tests")
import torch
from _util import make_net, golden, rel_err
from dquartic.model.model import DDIMDiffusionModel

g = golden("train_tiny.npz")
gg = golden("train_tiny_grads.npz")
net, P = make_net()
net.train()
d = DDIMDiffusionModel(net, device="cuda")
x0, c2, c1 = (torch.from_numpy(g[k]).cuda() for k in ("x0", "ms2_cond", "ms1_cond"))
noise = torch.from_numpy(g["noise"]).cuda(); t = torch.from_numpy(g["t"]).cuda()
net.zero_grad()
loss = d.train_step(x0, c2, c1, noise=(noise + 1) * 0.5, t=t)
loss.mean().backward()
print("loss", float(loss.mean()), float(g["loss"]))
rows = []
for k in P:
    if k.endswith("freqs"): continue
    ref = torch.from_numpy(gg["grad:" + k]); got = net._params[k].grad.cpu()
    e = float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
    cos = float(torch.dot(got.flatten(), ref.flatten()) / (got.norm() * ref.norm()).clamp_min(1e-30))
    rows.append((e, cos, k, float(ref.abs().max())))
rows.sort(reverse=True)
for r in rows[:40]:
    print("%.3e cos=%.6f %-45s refmax=%.3e" % r)
print("...")
for r in rows[-5:]:
    print("%.3e cos=%.6f %-45s refmax=%.3e" % r)
