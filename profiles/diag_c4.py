import importlib, os, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT); PKG="multimodal-fusion-based-pre-routing-timing-prediction-_b200"; sys.path.insert(0, os.path.join(ROOT, PKG))
importlib.import_module(PKG)
import Unet as U, tm_unet
from oracle import restate
torch.manual_seed(4)
net = U.UNet("max").train()
sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
x = torch.rand(2, 3, 256, 256)
P = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v) for k, v in sd.items()}
ref, _ = restate.unet_forward(P, x, "max")
g = torch.randn_like(ref)
names = [k for k, _ in net.named_parameters()]
gref = torch.autograd.grad(ref, [P[k] for k in names], g)
net = net.to("cuda")
for mode in ("bf16", "tf32", "tc3", "tf32x3"):
    tm_unet.MATH = mode
    net.zero_grad()
    out = net(x.cuda()); out.backward(g.cuda())
    errs = []
    for k, r in zip(names, gref):
        a = dict(net.named_parameters())[k].grad.cpu().double(); b = r.double()
        errs.append((float((a-b).norm()/b.norm()), k))
    o = float((out.cpu().double()-ref.double()).norm()/ref.double().norm())
    errs.sort(reverse=True)
    print(mode, "out relL2 %.2e" % o, "worst grads:", [(f"{e:.2e}", k) for e, k in errs[:3]], "median %.2e" % errs[len(errs)//2][0])
