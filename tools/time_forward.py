"""Device time of one CUDA-graph-replayed batched UNet forward (cond+uncond of B images).
Usage: python tools/time_forward.py [B=4] [alpha=1] [iters=20]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from instancediffusion_b200 import synthetic
from instancediffusion_b200.utils.model import set_alpha_scale
from instancediffusion_b200.weights import build_unet

B = int(sys.argv[1]) if len(sys.argv) > 1 else 4
alpha = float(sys.argv[2]) if len(sys.argv) > 2 else 1.0
iters = int(sys.argv[3]) if len(sys.argv) > 3 else 20
dev = torch.device("cuda:0")
model = build_unet("box", dev, seed=0)
gti = model.grounding_tokenizer_input
inp, uc = synthetic.make_sampler_inputs(gti, B, 8, 77, "box", mis=False, device=dev)
inp["timesteps"] = torch.full((B,), 601, dtype=torch.long, device=dev)
un = dict(x=inp["x"], timesteps=inp["timesteps"], context=uc)
set_alpha_scale(model, alpha)
with torch.no_grad():
    for _ in range(3):
        model.forward_batched([inp, un])
    torch.cuda.synchronize()
    s = torch.cuda.Event(enable_timing=True)
    e = torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        model.forward_batched([inp, un])
    e.record()
    torch.cuda.synchronize()
ms = s.elapsed_time(e) / iters
tf = 2 * B * (1.136 if alpha else 0.803)
print(f"forward(batch {2 * B}, alpha={alpha}) {ms:.2f} ms  ~{tf / ms * 1e3:.0f} TFLOP/s (F_min)")
