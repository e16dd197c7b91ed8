#!/usr/bin/env python
"""bench.py - SDF decoder queries/s on N B200s (BASELINE.json metric), plus roofline, accuracy against the frozen
oracle, end-to-end (host buffers through the C ABI) and a CPU-oracle baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N = 1 - a step = decode_grid(z, 256): BASELINE.json configs[1], one latent on a 256^3 grid (16,777,216 queries), bf16
operands / fp32 accumulate, fused tcgen05 kernel.  The same step is also timed with fp16 operands (the precision that meets
the north star's 2e-3 bound against the fp32 oracle), and both precisions are CHECKED against the oracle in the run
(`accuracy`).

N > 1 - a step = BASELINE.json configs[4], the north star's target case: ONE latent, 512^3 grid (134,217,728 queries), a
z-slab per rank, the sign-change mask fused (halo plane recomputed locally), every finished sub-slab pushed into all peers'
copies of a symmetric buffer by the copy engines over NVLink while the next one is decoded (sdfb_decode_grid_sharded); the
assembled grid is checked bit for bit against a single-GPU decode.  Total work is fixed => "strong" scaling.  The
collective-free weak-scaling number of round 1 (one 256^3 grid per rank) is kept as `independent_grids`.

`--impl reference`: the mounted reference has no source (/root/reference/README.md:1 is a title), so the "reference arm"
is the frozen CPU oracle (oracle/, a PyTorch fp32 restatement of the method) timed on the box's host cores on a bounded
sample of the same workload.
"""
from __future__ import annotations

import argparse
import glob
import json
import os
import re
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RES = 256
QUERIES = RES ** 3
RES5 = 512
# work per query (SURVEY.md section 8d / DESIGN.md): MACs issued to the tensor pipe with the
# latent folded into biases and L3 padded to N=256: 6 * 512^2 ; dense count as the oracle computes it
FLOP_TENSOR_PER_QUERY = 2 * 6 * 512 * 512          # 3,145,728
FLOP_DENSE_PER_QUERY = 3_671_040
DDPM_LATENTS = 4096
DDPM_FLOP_PER_LATENT_STEP = 2 * (512 * 1024 + 3 * 1024 * 1024 + 1024 * 256)   # 7,864,320 executed (hi/lo split of x: K = 512)
METRIC = "sdf_decoder_queries_per_s"
UNIT = "queries/s"
REF_BUDGET_S = 15.0
DUMP_DRAWS = 1 << 22            # seeded draws per dumped array: ~4 M distinct elements, at most 16 MiB of float32


def dump_sample(t, seed: int):
    """--dump-outputs: a fixed, seeded sample of `t`'s elements (flat order) as float32, so that two builds can be compared
    element for element without writing a whole 256^3 / 512^3 grid."""
    import numpy as np
    import torch
    drawn = np.zeros(t.numel(), dtype=bool)
    drawn[np.random.RandomState(seed).randint(0, t.numel(), DUMP_DRAWS, dtype=np.int64)] = True
    idx = np.flatnonzero(drawn)                                # distinct, in ascending order
    return t.reshape(-1)[torch.from_numpy(idx).to(t.device)].float().cpu().numpy()


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            p = json.load(f)
        return {"burst": float(p["bf16_tflops"]), "sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                "source": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"burst": 1590.0, "sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def read_ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one fused_decoder_kernel launch from the newest committed
    `ncu --set full` summary under profiles/ (r<N>_fused_decoder_ncu_full.csv); (None, why) when there is none."""
    best = None
    for path in glob.glob(os.path.join(ROOT, "profiles", "r*_fused_decoder_ncu_full.csv")):
        m = re.match(r"r(\d+)_", os.path.basename(path))
        if m and (best is None or int(m.group(1)) > best[0]):
            best = (int(m.group(1)), path)
    if best is None:
        return None, "no profiles/r*_fused_decoder_ncu_full.csv"
    total, seen = 0.0, 0
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    with open(best[1]) as f:
        for line in f:
            parts = line.strip().split(",")
            if len(parts) >= 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and parts[1] in scale:
                total += float(parts[2]) * scale[parts[1]]
                seen += 1
    if seen != 2:
        return None, f"{os.path.basename(best[1])} lacks the dram__bytes rows"
    return int(total), (f"dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full capture profiles/"
                        f"{os.path.basename(best[1])} (file mtime {time.strftime('%Y-%m-%dT%H:%M:%SZ', time.gmtime(os.path.getmtime(best[1])))}; "
                        "not re-measured in this run)")


class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index: int, period_s: float = 0.02):
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:                      # noqa: BLE001
            self.nv, self.err = None, repr(e)

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:                   # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:                       # noqa: BLE001
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_oracle_rate(target_s: float = 12.0):
    """Oracle (fp32 torch CPU) queries/s on a bounded sample: z-slabs of the 256^3 workload."""
    import torch
    import oracle
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    z = oracle.default_latent()
    oracle.decode_grid(z, RES, 0, 1)                      # warm-up: one plane (65,536 queries)
    t0 = time.perf_counter()
    oracle.decode_grid(z, RES, 0, 2)
    dt = time.perf_counter() - t0
    planes = max(2, min(RES, int(target_s / max(dt / 2, 1e-6))))
    t0 = time.perf_counter()
    oracle.decode_grid(z, RES, 0, planes)
    dt = time.perf_counter() - t0
    q = planes * RES * RES
    return {"value": q / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"planes [0,{planes}) of the 256^3 grid = {q} queries in {dt:.2f} s, torch {torch.__version__} fp32, "
                      f"{cores} threads (oracle/decoder.py; no reference source exists to time)"}


def cpu_ddpm_rate(n: int = 1024, steps: int = 250):
    """Oracle DDPM sampler (fp32 torch CPU) latents/s on a bounded sample: n latents x `steps` of the 1000 steps."""
    import numpy as np
    import torch
    import oracle
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    rs = np.random.RandomState(0)
    x_T = rs.standard_normal((n, 256)).astype(np.float32)
    noise = rs.standard_normal((steps, n, 256)).astype(np.float32)
    oracle.sample_latents(n, x_T, noise[:5], steps=5)
    t0 = time.perf_counter()
    oracle.sample_latents(n, x_T, noise, steps=steps)
    dt = time.perf_counter() - t0
    return {"value": n / (dt * 1000.0 / steps), "unit": "latents/s", "cores": cores, "kind": "port",
            "sample": f"{n} latents x {steps} of 1000 steps in {dt:.2f} s (scaled to 1000 steps), torch fp32, {cores} threads"}


def run_reference(args):
    """The reference arm: the CPU oracle on the host cores, on the same metric and workload as the GPU arm at this N.
    Honours --steps / --warmup up to a time budget (REF_BUDGET_S of timed work) and says what it clipped."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    steps_req, warm_req = max(1, args.steps), max(0, args.warmup)
    import torch
    import oracle
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    z = oracle.default_latent()
    res = RES if args.gpus <= 1 else RES5
    planes = 4 if res == RES else 1                       # 262,144 queries per step (= configs[0]'s count)
    q = planes * res * res
    t0 = time.perf_counter()
    oracle.decode_grid(z, res, 0, planes)                 # first call (thread pool start-up), also a rate estimate
    est = time.perf_counter() - t0
    warm = min(warm_req, max(0, int(3.0 / max(est, 1e-3))))
    for _ in range(warm):
        oracle.decode_grid(z, res, 0, planes)
    t0 = time.perf_counter()
    oracle.decode_grid(z, res, 0, planes)
    est = time.perf_counter() - t0
    steps = max(1, min(steps_req, int(REF_BUDGET_S / max(est, 1e-3))))
    t0 = time.perf_counter()
    for s in range(steps):
        zz = (s * planes) % res
        oracle.decode_grid(z, res, zz, zz + planes)
    dt = time.perf_counter() - t0
    value = q * steps / dt
    workload = ("decode_grid(z, 256): one latent, 256^3 grid (BASELINE configs[1])" if res == RES else
                "decode_grid_sharded(z, 512): one latent, 512^3 grid (BASELINE configs[4])")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
        "scaling": "weak" if args.gpus <= 1 else "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{workload}; each step a bounded sample of {planes} z-plane(s) = {q} queries",
                   "note": "the mounted reference has no source; this arm is the frozen CPU oracle on the host cores"},
        "clipped": {"steps_requested": steps_req, "steps_run": steps, "warmup_requested": warm_req, "warmup_run": warm,
                    "budget_s": REF_BUDGET_S, "why": "CPU arm bounded to ~15 s of timed work; the metric is a rate"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{steps} steps x {q} queries, torch {torch.__version__} fp32, {cores} threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def accuracy_block(pkg, dec, torch, np):
    """Checker leg (the oracle is allowed here): both tensor-core precisions against the fp32 oracle and against the oracle
    that emulates their operand rounding, on the committed golden nodes of the 256^3 / 64^3 grids plus 4096 seeded nodes."""
    import oracle
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "oracle_golden.npz")))
    z = oracle.default_latent()
    rs = np.random.RandomState(2024)
    extra = np.sort(rs.choice(QUERIES, 4096, replace=False)).astype(np.int64)
    c = oracle.axis_coords(RES)
    pts = np.stack([c[extra % RES], c[(extra // RES) % RES], c[extra // (RES * RES)]], axis=1)
    ref_extra = oracle.decoder_forward(z, pts)
    out = {}
    for prec, lowp in (("bf16", torch.bfloat16), ("fp16", torch.float16)):
        sdf = dec.decode_grid(z, RES, precision=prec)
        dec.check()
        flat = sdf.reshape(-1)
        got_g = flat[torch.from_numpy(g["sdf256_idx"]).to(flat.device)].cpu().numpy()
        got_e = flat[torch.from_numpy(extra).to(flat.device)].cpu().numpy()
        got = np.concatenate([got_g, got_e])
        ref = np.concatenate([g["sdf256_fp32"], ref_extra])
        d = np.abs(got.astype(np.float64) - ref)
        far = np.abs(ref) > 2e-3
        emu = oracle.decoder_forward_lowp(z, pts, lowp=lowp)
        de = np.abs(got_e.astype(np.float64) - emu)
        out[prec] = {"max_abs_vs_fp32": float(d.max()), "p99_vs_fp32": float(np.quantile(d, 0.99)),
                     "p50_vs_fp32": float(np.quantile(d, 0.5)),
                     "sign_agreement_where_abs_gt_2e-3": float(((got < 0) == (ref < 0))[far].mean()),
                     "within_north_star_2e-3": bool(d.max() < 2e-3),
                     "max_abs_vs_rounding_emulating_oracle": float(de.max()),
                     "p90_vs_rounding_emulating_oracle": float(np.quantile(de, 0.9)),
                     "p99_vs_rounding_emulating_oracle": float(np.quantile(de, 0.99)), "n": int(got.size)}
        del sdf
    sdf32 = dec.decode_grid(z, 64, precision="fp32").reshape(-1)
    got32 = sdf32[torch.from_numpy(g["sdf64_idx"]).to(sdf32.device)].cpu().numpy()
    out["fp32_path"] = {"max_abs_vs_fp32": float(np.abs(got32 - g["sdf64_fp32"]).max()), "within_north_star_1e-5":
                        bool(np.abs(got32 - g["sdf64_fp32"]).max() < 1e-5), "n": int(got32.size), "grid": "64^3 golden nodes"}
    out["oracle"] = ("oracle.decoder_forward (fp32 torch CPU) / decoder_forward_lowp on tests/golden sdf256_idx (256 nodes) + 4096 "
                     "seeded nodes of the 256^3 grid; north star: 2e-3 max-abs, >= 99.9 % sign agreement where |sdf| > 2e-3")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-accuracy", action="store_true", help="skip the oracle check of both precisions")
    ap.add_argument("--no-second-precision", action="store_true", help="do not time the other tensor-core precision")
    ap.add_argument("--no-config5", action="store_true", help="N > 1: time independent 256^3 grids only (round-1 headline)")
    ap.add_argument("--no-config4", action="store_true", help="skip the sample-then-decode leg (configs[3])")
    ap.add_argument("--no-ddpm", action="store_true", help="skip the latent-DDPM leg (second half of the metric)")
    ap.add_argument("--no-vjp", action="store_true", help="skip the latent-gradient leg (SURVEY 8f row N4)")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step legs (SURVEY 8f row N4)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the headline step returned in its last timed step to DIR/<name>.npy (float32, rank 0): a fixed "
                         "seeded sample of the sdf grid, and with the sharded 512^3 headline (N > 1) of its unpacked sign-change mask")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the GPU arm's outputs; the reference arm has none to compare")
        return run_reference(args)

    # stdout carries exactly one JSON line: anything libraries print there (NCCL's version banner, ...) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    # the CPU baselines run on rank 0 at N = 1 only, and BEFORE any GPU work (nothing waits for them on a GPU)
    cpu_base = cpu_ddpm = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_oracle_rate()
        if not args.no_ddpm:
            cpu_ddpm = cpu_ddpm_rate()

    import numpy as np
    import torch
    import torch.distributed as dist
    from __graft_entry__ import load_package

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = load_package()
    K, W = max(1, args.steps), max(3, args.warmup)
    dev = torch.device("cuda", local)
    dec = pkg.Decoder(pkg.synthetic.decoder_params(), device=dev, precision=args.precision)
    z_host = pkg.synthetic.latent(rank)                            # each rank: its own latent (independent grids)
    z = torch.from_numpy(z_host).to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)    # 256 MiB > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v: float) -> float:
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def time_grid(prec: str, steps: int, warm: int, clk=None):
        """`steps` timed decode_grid(z, 256) calls: (sum of per-step event times, max over ranks; mean kernel ms; the sdf
        of the last step)."""
        out = torch.empty((RES, RES, RES), dtype=torch.float32, device=dev)
        for _ in range(warm):
            dec.decode_grid(z, RES, out=out, precision=prec)
        barrier()
        kms = []
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i in range(steps):
            flush.fill_(float(i))                                  # evict L2 between timed iterations (untimed)
            ev[i][0].record()
            dec.decode_grid(z, RES, out=out, precision=prec)       # fold kernel + fused kernel on the current stream
            ev[i][1].record()
            ev[i][1].synchronize()
            kms.append(dec.last_kernel_ms())                       # events around the fused kernel itself; raises on a watchdog trip
        barrier()
        total = max_over_ranks(sum(a.elapsed_time(b) for a, b in ev))
        return total, statistics.mean(kms), out

    peaks = read_peaks()
    headline5 = world > 1 and not args.no_config5
    line = {}
    dumps = {}                                                     # --dump-outputs: name -> sampled float32 array

    # ---- decode_grid(z, 256) per rank: the N = 1 headline; at N > 1 the collective-free weak-scaling number
    with ClockSampler(local) as clk1:
        t_wall0 = time.perf_counter()
        Kg = K if not headline5 else max(3, min(K, 5))
        total_ms, k_ms, sdf_last = time_grid(args.precision, Kg, W)
        t_wall = time.perf_counter() - t_wall0
    if args.dump_outputs and rank == 0 and not headline5:
        dumps["sdf"] = dump_sample(sdf_last, 0)
    del sdf_last
    grid_value = world * QUERIES * Kg / (total_ms * 1e-3)
    achieved = QUERIES * FLOP_TENSOR_PER_QUERY / (k_ms * 1e-3) / 1e12
    traffic, traffic_src = read_ncu_traffic()
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peaks["burst"], "unit": "TFLOP/s",
                "frac": achieved / peaks["burst"], "traffic": traffic,
                "traffic_source": traffic_src + "; algorithmic bytes = 67,108,864 output bytes, part of which is still in L2 when the launch ends",
                "peak_kind": "burst bf16 matmul, " + peaks["source"],
                "frac_of_sustained": achieved / peaks["sustained"], "peak_sustained": peaks["sustained"],
                "kernel": "fused_decoder_kernel", "kernel_ms": k_ms, "workload": "decode_grid(z, 256), one launch = 16,777,216 queries",
                "flop_per_query_tensor_pipe": FLOP_TENSOR_PER_QUERY,
                "dense_equiv_tflops": QUERIES * FLOP_DENSE_PER_QUERY / (k_ms * 1e-3) / 1e12}

    # ---- the other tensor-core precision on the same step (fp16 operands meet the 2e-3 bound against the fp32 oracle)
    second = None
    if not args.no_second_precision:
        other = "fp16" if args.precision == "bf16" else "bf16"
        Ks = max(3, min(K, 10))
        t2, k2, _ = time_grid(other, Ks, 2)
        a2 = QUERIES * FLOP_TENSOR_PER_QUERY / (k2 * 1e-3) / 1e12
        second = {"dtype": other, "value": world * QUERIES * Ks / (t2 * 1e-3), "unit": UNIT, "steps": Ks, "ms_per_step": t2 / Ks,
                  "kernel_ms": k2, "achieved_tflops": a2, "frac_of_burst_peak": a2 / peaks["burst"],
                  "workload": "the same decode_grid(z, 256) step, same kernel instantiated for the other 16-bit operand type"}

    # ---- accuracy of both precisions against the frozen oracle, measured in this run (rank 0)
    accuracy = None
    if rank == 0 and not args.no_accuracy:
        try:
            accuracy = accuracy_block(pkg, dec, torch, np)
        except Exception as exc:                     # a checker leg must never cost the headline line
            accuracy = {"error": repr(exc)}
            print(f"bench.py: accuracy leg failed: {exc!r}", file=sys.stderr)

    # ---- end to end: numpy latent in, numpy sdf out through the host-buffer C-ABI call ----
    sdf_host = torch.empty((RES, RES, RES), dtype=torch.float32).pin_memory().numpy()
    for _ in range(2):
        dec.decode_grid_host(z_host, RES, out=sdf_host)
    barrier()
    Ke = max(3, min(K, 10))
    t0 = time.perf_counter()
    for _ in range(Ke):
        dec.decode_grid_host(z_host, RES, out=sdf_host)
    e2e_grid = world * QUERIES * Ke / max_over_ranks(time.perf_counter() - t0)
    checksum = float(np.float64(sdf_host[::16, ::16, ::16].sum()))
    # the same call with a pageable output array (what the INTEGRATION.md stub passes)
    sdf_page = np.empty((RES, RES, RES), dtype=np.float32)
    dec.decode_grid_host(z_host, RES, out=sdf_page)
    barrier()
    Kp = 3
    t0 = time.perf_counter()
    for _ in range(Kp):
        dec.decode_grid_host(z_host, RES, out=sdf_page)
    e2e_pageable = world * QUERIES * Kp / max_over_ranks(time.perf_counter() - t0)
    same_bits = bool(np.array_equal(sdf_page, sdf_host))
    del sdf_page

    # ---- BASELINE configs[4], the headline when N > 1: ONE latent, 512^3, z-slab per rank, fused mask, pushes overlapped
    cfg5 = None
    if headline5:
        del flush
        z5_host = pkg.synthetic.latent(0)
        z5 = torch.from_numpy(z5_host).to(dev)
        # the overlapped path needs CUDA IPC between the ranks' processes and a loadable NCCL; if any rank cannot set it up,
        # ALL ranks fall back to decode + torch.distributed all-gathers (decided collectively, so nobody waits alone)
        comm, why = None, ""
        try:
            if os.environ.get("SDFB_BENCH_NO_COMM"):          # exercises the fallback below on a box where the peer path works
                raise RuntimeError("peer-memory path switched off by SDFB_BENCH_NO_COMM")
            comm = pkg.Comm(dev)
            comm.decode_grid_sharded(dec, z5, RES5, mask=True)
            torch.cuda.synchronize()
        except Exception as exc:                     # noqa: BLE001
            comm, why = None, repr(exc)
            print(f"bench.py: peer-memory path unavailable on rank {rank}: {exc!r}", file=sys.stderr)
        okc = torch.tensor([1 if comm is not None else 0], device=dev)
        dist.all_reduce(okc, op=dist.ReduceOp.MIN)
        push_path = bool(okc.item())

        def cfg5_step(precision=None):
            if push_path:
                return comm.decode_grid_sharded(dec, z5, RES5, mask=True, precision=precision)
            if precision is None:
                return pkg.decode_grid_sharded(dec, z5, RES5, mask=True)
            z0_, z1_ = pkg.slab_range(RES5, rank, world)          # fallback in the other precision: this rank's slab only
            return dec.decode_grid(z5, RES5, z0_, z1_, mask=True, precision=precision)

        for _ in range(W):
            s5, m5 = cfg5_step()
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        with ClockSampler(local) as clk5:
            for i in range(K):
                barrier()
                ev[i][0].record()
                s5, m5 = cfg5_step()
                ev[i][1].record()
                ev[i][1].synchronize()
            barrier()
        dec.check()
        if args.dump_outputs and rank == 0:          # s5 / m5 of the push path are views: sampled before the next sharded decode
            dumps["sdf"] = dump_sample(s5, 0)
            dumps["mask"] = dump_sample(pkg.unpack_mask_blocks(m5, RES5) if push_path else m5, 1)
        step5 = [a.elapsed_time(b) for a, b in ev]
        total5 = max_over_ranks(sum(step5))
        med5 = max_over_ranks(statistics.median(step5))
        # bit identity: the assembled grid and mask on EVERY rank against this rank's own single-GPU decode of the whole grid
        ref_s, ref_m = dec.decode_grid(z5, RES5, mask=True)
        ok = bool(torch.equal(s5, ref_s)) and bool(torch.equal(pkg.unpack_mask_blocks(m5, RES5) if push_path else m5, ref_m))
        okt = torch.tensor([int(ok)], device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        active = int(ref_m.sum().item())
        chk = float(s5[::32, ::32, ::32].double().sum().item())
        del ref_s, ref_m
        # the same step in the other 16-bit operand type (fp16 meets the 2e-3 bound against the fp32 oracle)
        other5 = "fp16" if args.precision == "bf16" else "bf16"
        t_other = []
        for i in range(1 + 4):
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            so, mo = cfg5_step(other5)
            b.record()
            b.synchronize()
            if i:
                t_other.append(a.elapsed_time(b))
        dec.check()
        other_ms = max_over_ranks(statistics.mean(t_other))
        other_chk = float(so[::32, ::32, ::32].double().sum().item()) if push_path else None
        del so, mo
        # the torch.distributed path of round 1 (decode, then NCCL all-gathers of sdf and uint8 mask), for comparison
        t_nccl = []
        for _ in range(3):
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            s5b, m5b = pkg.decode_grid_sharded(dec, z5, RES5, mask=True)
            b.record()
            b.synchronize()
            t_nccl.append(a.elapsed_time(b))
        del s5b, m5b
        # end to end with host buffers: every rank's slab (+ mask) through decode_grid_host, the host side holds the grid
        z0, z1 = pkg.slab_range(RES5, rank, world)
        slab_host = torch.empty((z1 - z0, RES5, RES5), dtype=torch.float32).pin_memory().numpy()
        dec.decode_grid_host(z5_host, RES5, z0, z1, mask=True, out=slab_host)
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            _, mh = dec.decode_grid_host(z5_host, RES5, z0, z1, mask=True, out=slab_host)
        e2e5 = RES5 ** 3 * 3 / max_over_ranks(time.perf_counter() - t0)
        per_gpu_tflops = (RES5 ** 3 / world) * FLOP_TENSOR_PER_QUERY / (total5 / K * 1e-3) / 1e12
        ideal_ms = k_ms * (RES5 ** 3 / world + RES5 * RES5) / QUERIES          # slab + halo plane at the measured single-GPU kernel rate
        cfg5 = {"ms_per_step": total5 / K, "median_ms": med5, "queries_per_s": RES5 ** 3 * K / (total5 * 1e-3),
                "tflops_per_gpu_incl_mask_and_assembly": per_gpu_tflops, "frac_of_burst_peak_per_gpu": per_gpu_tflops / peaks["burst"],
                "one_gpu_ideal_ms": ideal_ms, "efficiency_vs_1gpu_ideal": ideal_ms / (total5 / K),
                "bit_identical": bool(okt.item()), "active_cells": active, "sdf_checksum": chk,
                "path": "sdfb_decode_grid_sharded (copy-engine pushes into CUDA-IPC peer buffers, overlapped)" if push_path
                        else "fallback: decode, then torch.distributed all-gathers (" + why[:120] + ")",
                "torch_distributed_path_ms": max_over_ranks(statistics.median(t_nccl)),
                "second_precision": {"dtype": other5, "ms_per_step": other_ms, "steps": len(t_other), "sdf_checksum": other_chk,
                                     "frac_of_burst_peak_per_gpu": (RES5 ** 3 / world) * FLOP_TENSOR_PER_QUERY / (other_ms * 1e-3) / 1e12 / peaks["burst"]},
                "e2e_host_slabs_queries_per_s": e2e5, "e2e_d2h_bytes_per_rank": int(slab_host.nbytes + mh.nbytes),
                "clocks": clk5.summary()}
        del s5, m5

    # ---- second half of the metric: latent-DDPM latents/s (BASELINE configs[3]: 4096 latents, 1000 steps) ----
    ddpm_line = None
    if not args.no_ddpm:
        try:
            n_lat, T = DDPM_LATENTS, 1000
            sampler = pkg.LatentDDPM(pkg.synthetic.ddpm_params(), device=dev, precision=args.precision)
            g = torch.Generator(device=dev).manual_seed(100 + rank)
            x_T = torch.randn((n_lat, 256), generator=g, device=dev)
            noise = torch.randn((T, n_lat, 256), generator=g, device=dev)           # 4.2 GB explicit noise stream in HBM
            dd_ms = []
            for i in range(1 + 3):                                                   # 1 warm-up + 3 timed full samplings
                barrier()
                x0 = sampler.sample_latents(n_lat, x_T=x_T, noise=noise, steps=T)
                if i:
                    dd_ms.append(sampler.last_kernel_ms())
            dd_ms_max = max_over_ranks(statistics.mean(dd_ms))
            flop = n_lat * T * DDPM_FLOP_PER_LATENT_STEP
            ddpm_line = {"metric": "ddpm_latents_per_s", "value": world * n_lat / (dd_ms_max * 1e-3), "unit": "latents/s",
                         "workload": f"sample_latents({n_lat}) per GPU: MLP denoiser 4x1024, latent 256, {T} steps, explicit noise "
                                     "stream resident in HBM; ONE persistent kernel per call",
                         "ms_per_sampling": dd_ms_max, "us_per_step": dd_ms_max * 1e3 / T,
                         "kernel": "ddpm_sample_kernel", "achieved_tflops": flop / (dd_ms_max * 1e-3) / 1e12,
                         "flop_per_latent_step": DDPM_FLOP_PER_LATENT_STEP, "gpu_launches_per_sampling": 2,
                         "x0_abs_max": float(x0.abs().max().item())}
            ddpm_line["frac_of_burst_peak"] = ddpm_line["achieved_tflops"] / peaks["burst"]
            del noise
            # sample_latents(n) as the north star spells it - no stream argument: noise generated in the kernel
            # (Philox4x32-10), device-timed, then end to end through the host-buffer call (x_0 [n,256] comes back)
            sd_ms = []
            for i in range(1 + 3):
                barrier()
                xs0 = sampler.sample_latents(n_lat, steps=T, seed=7 + rank)
                if i:
                    sd_ms.append(sampler.last_kernel_ms())
            sd = max_over_ranks(statistics.mean(sd_ms))
            ddpm_line["seeded"] = {"value": world * n_lat / (sd * 1e-3), "unit": "latents/s", "ms_per_sampling": sd,
                                   "noise": "generated in the update epilogue (Philox4x32-10 + Box-Muller), no noise stream in memory",
                                   "x0_abs_max": float(xs0.abs().max().item())}
            sampler.sample_latents_seeded_host(n_lat, 7 + rank, steps=T)
            barrier()
            t0 = time.perf_counter()
            for _ in range(3):
                xh = sampler.sample_latents_seeded_host(n_lat, 7 + rank, steps=T)
            e2 = max_over_ranks((time.perf_counter() - t0) / 3)
            ddpm_line["e2e"] = {"value": world * n_lat / e2, "unit": "latents/s", "h2d_bytes_per_step": 0,
                                "d2h_bytes_per_step": int(xh.nbytes),
                                "api": "LatentDDPM.sample_latents_seeded_host -> sdfb_ddpm_sample_philox_host (x_T and noise generated on the device, x_0 returned to the host)"}
            # config 4's per-GPU share on 8 GPUs: 512 latents
            s512 = []
            for i in range(1 + 3):
                barrier()
                sampler.sample_latents(512, steps=T, seed=11 + rank)
                if i:
                    s512.append(sampler.last_kernel_ms())
            m512 = max_over_ranks(statistics.mean(s512))
            ddpm_line["n512"] = {"ms_per_sampling": m512, "latents_per_s": world * 512 / (m512 * 1e-3),
                                 "achieved_tflops": 512 * T * DDPM_FLOP_PER_LATENT_STEP / (m512 * 1e-3) / 1e12}
            if cpu_ddpm is not None:
                ddpm_line["cpu_baseline"] = cpu_ddpm
            del sampler
        except Exception as exc:                     # an optional leg must never cost the headline line
            ddpm_line = {"error": repr(exc)}
            print(f"bench.py: optional leg failed: {exc!r}", file=sys.stderr)

    # ---- BASELINE configs[3], one GPU's share when it is spread over 8: 512 of the 4096 latents are sampled (1000 steps,
    # noise generated in the kernel), scaled into the decoder's latent range, and each is decoded on a 128^3 grid (64 shapes
    # per call into a reused buffer; 34 GB of sdf in total for the full config, so the fields are consumed as they are produced)
    cfg4 = None
    if not args.no_config4:
        try:
            n4, res4 = 512, 128
            smp = pkg.LatentDDPM(pkg.synthetic.ddpm_params(), device=dev, precision=args.precision)
            buf4 = torch.empty((64, res4, res4, res4), dtype=torch.float32, device=dev)
            lat4 = smp.sample_latents(n4, seed=1000 + rank) * pkg.DDPM_LATENT_SCALE
            dec.decode_grid_batch(lat4[:64], res4, out=buf4)
            barrier()
            a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            a.record()
            lat4 = smp.sample_latents(n4, seed=1000 + rank) * pkg.DDPM_LATENT_SCALE
            b.record()
            inside = []
            for i0 in range(0, n4, 64):
                dec.decode_grid_batch(lat4[i0:i0 + 64], res4, out=buf4)
                if i0 == 0:
                    inside = [float((buf4[j] < 0).float().mean().item()) for j in range(4)]   # untimed-size check: real surfaces
            c.record()
            c.synchronize()
            dec.check()
            t4 = torch.tensor([a.elapsed_time(b), b.elapsed_time(c)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t4, op=dist.ReduceOp.MAX)
            q4 = n4 * res4 ** 3
            cfg4 = {"workload": f"per GPU: sample_latents({n4}) (1000 steps, in-kernel noise), x DDPM_LATENT_SCALE, then decode_grid_batch of the "
                                f"{n4} samples at {res4}^3 (64 per call); {world} GPUs cover {world * n4} latents (BASELINE configs[3] = 4096 latents on 8 GPUs)",
                    "ddpm_ms": float(t4[0].item()), "decode_ms": float(t4[1].item()), "total_ms": float(t4.sum().item()),
                    "decode_queries_per_s": world * q4 / (float(t4[1].item()) * 1e-3),
                    "decode_tflops_per_gpu": q4 * FLOP_TENSOR_PER_QUERY / (float(t4[1].item()) * 1e-3) / 1e12,
                    "inside_fraction_first_4_shapes": inside}
            del buf4, smp, lat4
        except Exception as exc:                     # an optional leg must never cost the headline line
            cfg4 = {"error": repr(exc)}
            print(f"bench.py: optional leg failed: {exc!r}", file=sys.stderr)

    # ---- SURVEY 8f row N4: latent gradient (auto-decoder fitting) through the forward + backward instance of the fused
    # kernel, next to the fp32 path on a sample of the same points
    vjp = None
    if not args.no_vjp:
        try:
            n_v = 1 << 22
            gv = torch.Generator(device=dev).manual_seed(7 + rank)
            pts = torch.rand((n_v, 3), generator=gv, device=dev) * 2 - 1
            up = torch.randn(n_v, generator=gv, device=dev) / n_v
            zv = torch.from_numpy(pkg.synthetic.latent(rank)).to(dev)
            dec.latent_vjp(zv, pts, up, precision=args.precision)
            barrier()
            ms_v = []
            for _ in range(3):
                dec.latent_vjp(zv, pts, up, precision=args.precision)
                ms_v.append(dec.last_kernel_ms())
            n32 = 1 << 17
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dec.latent_vjp(zv, pts[:n32], up[:n32], precision="fp32")
            a.record()
            dec.latent_vjp(zv, pts[:n32], up[:n32], precision="fp32")
            b.record()
            b.synchronize()
            kv = max_over_ranks(statistics.median(ms_v))
            vjp = {"workload": f"per GPU: latent_vjp over {n_v} random points, precision {args.precision} (one launch of "
                               "fused_decoder_kernel<., BWD>: forward + 13 backward passes per tile)",
                   "kernel_ms": kv, "points_per_s": world * n_v / (kv * 1e-3),
                   "achieved_tflops_per_gpu": n_v * 2 * FLOP_TENSOR_PER_QUERY / (kv * 1e-3) / 1e12,
                   "fp32_path_points_per_s": n32 / (a.elapsed_time(b) * 1e-3)}
            vjp["frac_of_burst_peak"] = vjp["achieved_tflops_per_gpu"] / peaks["burst"]
            del pts, up
        except Exception as exc:                     # an optional leg must never cost the headline line
            vjp = {"error": repr(exc)}
            print(f"bench.py: optional leg failed: {exc!r}", file=sys.stderr)

    # ---- SURVEY 8f rows N1 / N2: surface extraction at 512^3 on ONE GPU - dense decode + marching cubes against the two-level
    # sparse decode (every node at most once) feeding the same dense marching-cubes kernels; identical triangle soups
    sparse = None
    if world == 1 and not args.no_vjp:
        try:
            zs_ = torch.from_numpy(pkg.synthetic.latent(0)).to(dev)
            dec.extract_surface_sparse(zs_, RES5)
            torch.cuda.synchronize()
            a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            a.record()
            tri_s, st_s = dec.extract_surface_sparse(zs_, RES5, return_stats=True)
            b.record()
            tri_d = dec.extract_surface(zs_, RES5)
            c.record()
            c.synchronize()
            dec.extract_surface_sparse(zs_, RES5, local_floor=0.5)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            tri_l, st_l = dec.extract_surface_sparse(zs_, RES5, local_floor=0.5, return_stats=True)
            e1.record()
            e1.synchronize()
            sparse = {"workload": "extract_surface_sparse(z, 512) vs extract_surface(z, 512) on one GPU (decode + marching cubes)",
                      "sparse_ms": a.elapsed_time(b), "dense_ms": b.elapsed_time(c), "triangles": int(tri_s.shape[0]),
                      "identical_triangle_soup": bool(tri_s.shape == tri_d.shape and torch.equal(tri_s, tri_d)),
                      "queries": st_s["queries"], "dense_queries": st_s["dense_queries"],
                      "fewer_queries_x": st_s["dense_queries"] / max(st_s["queries"], 1),
                      "local_slopes": {"what": "second level bounded by each block's own measured slope (floor 0.5 x the global bound)",
                                       "sparse_ms": e0.elapsed_time(e1), "queries": st_l["queries"],
                                       "fewer_queries_x": st_l["dense_queries"] / max(st_l["queries"], 1),
                                       "identical_triangle_soup": bool(tri_l.shape == tri_d.shape and torch.equal(tri_l, tri_d))}}
            del tri_s, tri_d, tri_l
        except Exception as exc:                     # an optional leg must never cost the headline line
            sparse = {"error": repr(exc)}
            print(f"bench.py: optional leg failed: {exc!r}", file=sys.stderr)

    # ---- SURVEY 8f row N4, second half: training steps (decoder weight gradients; DDPM training step), when built
    train = None
    if not args.no_train and hasattr(pkg, "bench_training_legs"):
        try:
            train = pkg.bench_training_legs(dec, dev, rank, world, args.precision, max_over_ranks, barrier, peaks)
        except Exception as exc:                     # an optional leg must never cost the headline line
            train = {"error": repr(exc)}
            print(f"bench.py: optional leg failed: {exc!r}", file=sys.stderr)

    if rank == 0:
        if headline5:
            value, ms_step, steps_out = cfg5["queries_per_s"], cfg5["ms_per_step"], K
            config = {"workload": f"decode_grid_sharded(z, 512, mask=True) on {world} GPUs (BASELINE configs[4]): ONE latent, 512^3 grid = "
                                  "134,217,728 queries, one z-slab per rank, fused sign-change mask with locally recomputed halo plane, every "
                                  "finished sub-slab pushed into all peers' copies of a symmetric buffer by the copy engines over NVLink while the "
                                  "next is decoded (sdfb_decode_grid_sharded), rank barrier at both ends; seeded random-init decoder 8x512, latent 256",
                      "l2": "each step writes 512 MiB of sdf per rank (> 126 MB L2) and every rank re-reads nothing; no separate flush",
                      "timing": "CUDA events per step on the launching stream (barrier + synchronize before each), summed, max over ranks",
                      "parallelism": f"z-slabs over {world} ranks; the only inter-GPU traffic is the assembly of the slabs"}
            scaling, clocks = "strong", cfg5["clocks"]
            e2e = {"value": cfg5["e2e_host_slabs_queries_per_s"], "unit": UNIT, "h2d_bytes_per_step": 1024,
                   "d2h_bytes_per_step": cfg5["e2e_d2h_bytes_per_rank"], "steps": 3,
                   "api": "per rank: Decoder.decode_grid_host(z, 512, z0, z1, mask=True) -> sdfb_decode_grid_host on its own slab "
                          "(numpy latent in, pinned numpy slab + uint8 mask out; bytes are per rank)"}
            own = RES5 // world                      # planes per rank; sub-slabs of >= 8 planes (2^21 queries), at most 16 of them
            sub = max(8, -(-(own + 1) // 16))
            launches = K * (2 * (-(-own // sub)) + 2)    # per rank and step: sub-slabs x (fold + fused kernel) + the two mask kernels
        else:
            value, ms_step, steps_out = grid_value, total_ms / Kg, Kg
            config = {"workload": "decode_grid(z, 256): one latent per GPU, 256^3 grid = 16,777,216 queries "
                                  "(BASELINE configs[1]); seeded random-init decoder 8x512, latent 256",
                      "l2": "256 MiB buffer written between timed iterations (L2 flush, untimed)",
                      "timing": "CUDA events per step on the launching stream, summed, max over ranks",
                      "parallelism": f"dp{world} (independent latents, no data-path collective)"}
            scaling, clocks = "weak", clk1.summary()
            e2e = {"value": e2e_grid, "unit": UNIT, "h2d_bytes_per_step": 1024, "d2h_bytes_per_step": QUERIES * 4,
                   "steps": Ke, "api": "Decoder.decode_grid_host -> sdfb_decode_grid_host (numpy in, pinned numpy out)",
                   "checksum": checksum}
            launches = 2 * Kg
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps_out, "warmup": W,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic", "config": config, "clocks": clocks, "e2e": e2e,
            "gpu_launches": launches, "roofline": roofline,
            "e2e_pageable": {"value": e2e_pageable, "unit": UNIT, "steps": Kp, "same_bits_as_pinned": same_bits,
                             "api": "the same sdfb_decode_grid_host call writing into a pageable numpy array (decode_grid(z, 256) per rank)"},
            "wall_s_timed_region": t_wall,
        }
        if headline5:
            line["config5_512cubed_sharded"] = cfg5
            line["independent_grids"] = {"value": grid_value, "unit": UNIT, "ms_per_step": total_ms / Kg, "steps": Kg,
                                         "e2e": e2e_grid, "clocks": clk1.summary(),
                                         "workload": "decode_grid(z, 256) per rank, independent latents (round 1's weak-scaling headline)"}
        if second is not None:
            line["second_precision"] = second
        if accuracy is not None:
            line["accuracy"] = accuracy
        if cfg4 is not None:
            line["config4_sample_then_decode"] = cfg4
        if vjp is not None:
            line["latent_gradient"] = vjp
        if train is not None:
            line["training"] = train
        if sparse is not None:
            line["sparse_extraction"] = sparse
        if ddpm_line is not None:
            line["ddpm"] = ddpm_line
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        elif world > 1:
            line["cpu_baseline_note"] = "timed on rank 0 at N = 1 only (see the N = 1 line)"
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dumps.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
