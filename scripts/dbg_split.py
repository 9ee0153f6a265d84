"""fp32 mode: the inference forward (fp16-split tensor-core kernel) against the training forward (bf16-split layer GEMMs) and an
fp64 torch MLP on the same weights."""
import os, sys, json, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import nerf_sandbox_b200 as nsb
from oracle import nerf_oracle as O
DEV = torch.device("cuda", 0)
T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
net = nsb.NeRF(63, 27, mode="fp32").to(DEV)
with torch.no_grad(): net.sigma_out.bias.fill_(0.3)
rng = np.random.default_rng(0)
Q = 20000
ep = T(O.positional_encode(rng.uniform(-4, 4, (Q, 3)).astype(np.float32), 10)); ed = T(O.positional_encode(O._normalize(rng.standard_normal((Q, 3)).astype(np.float32)), 4))
with torch.no_grad():
    a = net(ep, ed)                      # no stash -> fp16-split inference kernel
b = net(ep, ed)                          # grad enabled -> stash -> bf16-split GEMM chain
# fp64 reference
sd = {k: v.double() for k, v in net.state_dict().items()}
h = ep.double()
for l in range(8):
    x = torch.cat([h, ep.double()], -1) if l == 4 else h
    h = torch.relu(x @ sd[f"mlp.{l}.weight"].T + sd[f"mlp.{l}.bias"])
sig = h @ sd["sigma_out.weight"].T + sd["sigma_out.bias"]
feat = h @ sd["feature.weight"].T + sd["feature.bias"]
c = torch.relu(torch.cat([feat, ed.double()], -1) @ sd["color_fc.weight"].T + sd["color_fc.bias"])
ref = torch.cat([c @ sd["color_out.weight"].T + sd["color_out.bias"], sig], -1)
err = lambda x: (float((x.double() - ref).abs().max()), float((x.double() - ref).norm() / ref.norm()))
print(json.dumps({"split_vs_fp64": err(a), "train_fwd_vs_fp64": err(b.detach()), "mode": "fp32"}))
