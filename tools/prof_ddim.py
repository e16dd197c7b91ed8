#!/usr/bin/env python
"""Device time of the fused sampler on respaced schedules: the full 1000-step DDPM chain, DDIM at S = 25, 50, 100 with
eta = 0 and 1, and DDIM inversion at S = 50, for n = 512 and 4096 latents (seeded, bf16).  Each figure is the median of
`reps` timed calls after one warm-up call of the same shape (CUDA events around the one persistent launch).

    usage: python tools/prof_ddim.py [reps]"""
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from __graft_entry__ import load_package


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return f"{name}, power limit / max SM clock: {q.stdout.strip()}"
    except (OSError, subprocess.SubprocessError):
        return f"{name}, power limit: not available"


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    if not torch.cuda.is_available():
        raise SystemExit("prof_ddim.py needs a CUDA device")
    pkg = load_package()
    m = pkg.LatentDDPM(pkg.synthetic.ddpm_params(), device="cuda:0", precision="bf16")
    print(gpu_info())
    print(f"{'n':>5} {'run':<22} {'steps':>5} {'ms':>9} {'us/step':>8}")
    for n in (512, 4096):
        x0 = torch.randn((n, 256), generator=torch.Generator(device="cuda").manual_seed(1), device="cuda") * 0.5
        runs = [("ddpm", 1000, lambda: m.sample_latents(n, seed=3))]
        for S in (25, 50, 100):
            for eta in (0.0, 1.0):
                runs.append((f"ddim eta={eta:g}", S, lambda S=S, eta=eta: m.sample_latents_ddim(n, steps=S, eta=eta, seed=3)))
        runs.append(("ddim inversion", 50, lambda: m.invert_latents_ddim(x0, steps=50)))
        for name, steps, fn in runs:
            fn()
            m.last_kernel_ms()
            ts = []
            for _ in range(reps):
                fn()
                ts.append(m.last_kernel_ms())
            ms = statistics.median(ts)
            print(f"{n:>5} {name:<22} {steps:>5} {ms:>9.3f} {ms * 1e3 / steps:>8.2f}   (min {min(ts):.3f}, max {max(ts):.3f})", flush=True)
    m.close()


if __name__ == "__main__":
    main()
