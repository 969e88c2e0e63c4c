"""Is the VGG bias-gradient difference a GPU-vs-CPU library difference?  Plain torch modules only (no b200asr kernels)."""
import os, sys, numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import golden_params
g = dict(np.load(os.path.join(ROOT, "tests", "golden", "model_vgg.npz")))
P = golden_params(g, "vgg")
def build():
    c0, c1 = 64, 128
    ext = torch.nn.Sequential(
        torch.nn.Conv2d(1, c0, 3, 1, 1), torch.nn.ReLU(), torch.nn.Conv2d(c0, c0, 3, 1, 1), torch.nn.ReLU(), torch.nn.MaxPool2d(2, 2),
        torch.nn.Conv2d(c0, c1, 3, 1, 1), torch.nn.ReLU(), torch.nn.Conv2d(c1, c1, 3, 1, 1), torch.nn.ReLU(), torch.nn.MaxPool2d(2, 2))
    sd = {k[len("encoder.layers.0.extractor."):]: v for k, v in P.items() if k.startswith("encoder.layers.0.extractor.")}
    ext.load_state_dict(sd)
    return ext
feat = torch.from_numpy(g["feat"])
rem = feat.shape[1] % 4
if rem: feat = feat[:, :-rem].contiguous()
B, T, D = feat.shape
inC = D // 40
x = feat.view(B, T, inC, 40).transpose(1, 2).contiguous()
print("input", tuple(x.shape), "biases nonzero:", [float(v.abs().max()) for k, v in build().state_dict().items() if k.endswith("bias")])
torch.manual_seed(0)
res = {}
for name, dev, cudnn in (("cpu", "cpu", True), ("cuda", "cuda", True), ("cuda-nocudnn", "cuda", False)):
    torch.backends.cudnn.enabled = cudnn
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    m = build().to(dev)
    xi = x.detach().clone().to(dev).requires_grad_(True)
    y = m(xi)
    if "dy" not in res: res["dy"] = torch.randn(y.shape)
    y.backward(res["dy"].to(dev))
    res[name] = {k: p.grad.detach().cpu() for k, p in m.named_parameters()}
    res[name]["y"] = y.detach().cpu(); res[name]["dx"] = xi.grad.detach().cpu()
print("zeros in y(cpu): %d of %d" % (int((res["cpu"]["y"] == 0).sum()), res["cpu"]["y"].numel()))
for name in ("cuda", "cuda-nocudnn"):
    for k in res["cpu"]:
        a, b = res[name][k], res["cpu"][k]
        print("%-14s %-10s max|cpu| %.3e  max|diff| %.3e" % (name, k, float(b.abs().max()), float((a - b).abs().max())))
