#!/usr/bin/env python
"""Small end-to-end run of every kernel, meant to be wrapped in compute-sanitizer (one tool per gpurun call):
    compute-sanitizer --tool memcheck python tools/sanitize_small.py"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from __graft_entry__ import load_package

pkg = load_package()
dec = pkg.Decoder(pkg.synthetic.decoder_params(), device="cuda:0")
z = pkg.synthetic.latent(0)
for prec in ("bf16", "fp16", "fp32"):
    sdf, mask = dec.decode_grid(z, 24, 3, 11, mask=True, precision=prec)
    pts = torch.rand((301, 3), device="cuda") * 2 - 1
    out = dec(z, pts, precision=prec)
    torch.cuda.synchronize()
    print(prec, float(sdf.sum()), int(mask.sum()), float(out.sum()))
h, m = dec.decode_grid_host(z, 24, 3, 11, mask=True)
pts = torch.rand((777, 3), device="cuda") * 2 - 1            # latent gradient: fp32 path, backward instance, loss mode
up = torch.randn(777, device="cuda")
for prec in ("fp32", "bf16", "fp16"):
    g, y = dec.latent_vjp(z, pts, up, precision=prec)
    torch.cuda.synchronize()
    print("vjp", prec, float(g.sum()), float(y.sum()))
    if prec != "fp32":
        loss, g = dec.fit_loss_grad(z, pts, torch.zeros(777, device="cuda"), precision=prec)
        torch.cuda.synchronize()
        print("fit", prec, float(loss), float(g.sum()))
sdf, signs, mw = dec.decode_grid_bits(z, 24, mask=True)
tri = dec.extract_surface(z, 24)
tri_s = dec.extract_surface_sparse(z, 33)
print("surface", tuple(tri.shape), tuple(tri_s.shape))
ddpm = pkg.LatentDDPM(pkg.synthetic.ddpm_params(), device="cuda:0")
rs = np.random.RandomState(0)
x_T = rs.standard_normal((37, 256)).astype(np.float32)
noise = rs.standard_normal((3, 37, 256)).astype(np.float32)
for prec in ("bf16", "fp16", "fp32"):
    x = ddpm.sample_latents(37, x_T=x_T, noise=noise, steps=3, precision=prec)
    e = ddpm.denoise(x_T, 2, precision=prec)
    s = ddpm.sample_latents(300, steps=3, seed=5, precision=prec)
    torch.cuda.synchronize()
    print(prec, float(x.sum()), float(e.sum()), float(s.sum()))
print("done")
