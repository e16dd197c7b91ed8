#!/usr/bin/env python
"""End-to-end demo of the hot path on one GPU: sample latents with the fused DDPM kernel, decode one of them
(or the synthetic default latent) on a res^3 grid, extract the zero level set and write it as a Wavefront OBJ.

    python tools/demo.py [--res 128] [--out shape.obj] [--sampled [--ddim S]] [--sparse] [--fit N]

--ddim S samples with S respaced DDIM steps (eta = 0) instead of the 1000-step DDPM chain.

--fit N closes the loop: N SDF samples of the decoded shape are fitted by a FRESH latent (auto-decoder inference, one
forward + backward launch of the fused kernel per Adam step) and the refitted shape is what gets meshed.

Weights are seeded random-init (there are no checkpoints: the upstream repository has no code), so the
default latent gives a blob-like surface and a *sampled* latent usually gives an empty or saturated field."""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from __graft_entry__ import load_package


def write_obj(path, verts, faces):
    with open(path, "w") as f:
        f.write(f"# {verts.shape[0]} vertices, {faces.shape[0]} triangles\n")
        np.savetxt(f, verts, fmt="v %.7g %.7g %.7g")
        np.savetxt(f, faces + 1, fmt="f %d %d %d")
    return verts.shape[0], faces.shape[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=128)
    ap.add_argument("--out", default="shape.obj")
    ap.add_argument("--sampled", action="store_true", help="decode a latent drawn by the DDPM sampler instead of the synthetic one")
    ap.add_argument("--ddim", type=int, default=0, metavar="S", help="with --sampled: S deterministic DDIM steps instead of 1000 DDPM steps")
    ap.add_argument("--sparse", action="store_true", help="sparse extraction (decode only near the surface)")
    ap.add_argument("--fit", type=int, default=0, metavar="N", help="refit the shape from N of its own SDF samples (tensor-pipe latent fitting)")
    ap.add_argument("--fit-steps", type=int, default=400)
    args = ap.parse_args()
    pkg = load_package()
    dec = pkg.Decoder(pkg.synthetic.decoder_params())
    if args.sampled:
        ddpm = pkg.LatentDDPM(pkg.synthetic.ddpm_params(), precision="bf16")
        t0 = time.perf_counter()
        if args.ddim > 0:
            z = ddpm.sample_latents_ddim(256, steps=args.ddim, eta=0.0, seed=1)[0]
        else:
            z = ddpm.sample_latents(256, seed=1)[0]
        how = f"{args.ddim} DDIM steps" if args.ddim > 0 else "1000 DDPM steps"
        print(f"sampled 256 latents ({how}) in {ddpm.last_kernel_ms():.1f} ms (kernel), {1e3 * (time.perf_counter() - t0):.1f} ms (call)")
    else:
        z = torch.from_numpy(pkg.synthetic.latent(0)).cuda()
    if args.fit > 0:
        g = torch.Generator(device="cuda").manual_seed(0)
        pts = torch.rand((args.fit, 3), generator=g, device="cuda") * 2 - 1
        tgt = dec(z, pts, precision="fp32")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        z_fit, loss = dec.fit_latent(pts, tgt, steps=args.fit_steps, lr=1e-2, reg=0.0, precision="bf16")
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        held = torch.rand((20000, 3), generator=g, device="cuda") * 2 - 1
        err = float((torch.clamp(dec(z_fit, held, precision="fp32"), -0.1, 0.1) - torch.clamp(dec(z, held, precision="fp32"), -0.1, 0.1)).abs().mean())
        print(f"refitted a fresh latent to {args.fit} SDF samples: {args.fit_steps} Adam steps in {1e3 * dt:.1f} ms "
              f"({1e3 * dt / args.fit_steps:.3f} ms/step), train loss {loss:.5f}, held-out clamped-L1 {err:.5f}")
        z = z_fit
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if args.sparse:
        verts, faces = dec.extract_surface_sparse(z, args.res, indexed=True)
    else:
        verts, faces = dec.extract_surface(z, args.res, indexed=True)
    torch.cuda.synchronize()
    print(f"{'sparse' if args.sparse else 'dense'} extraction at {args.res}^3: {faces.shape[0]} triangles, {verts.shape[0]} vertices "
          f"(welded on the GPU) in {1e3 * (time.perf_counter() - t0):.1f} ms")
    nv, nf = write_obj(args.out, verts.cpu().numpy(), faces.cpu().numpy())
    print(f"wrote {args.out}: {nv} vertices, {nf} faces")


if __name__ == "__main__":
    main()
