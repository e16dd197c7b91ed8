"""bench.py's reference arm (the CPU oracle on the host cores) runs without a GPU: one short step here guards the
JSON contract of that arm; the keys of the GPU arm's line are checked on a saved line from profiles/, and its --dump-outputs
files on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config"}


def test_reference_arm_prints_one_json_line():
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["metric"] == "sdf_decoder_queries_per_s"
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_saved_gpu_line_has_the_contract_keys():
    with open(os.path.join(ROOT, "profiles", "r1_bench_n1.json")) as f:
        d = json.loads([ln for ln in f if ln.startswith("{")][-1])
    assert BASE_KEYS <= set(d)
    assert {"clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"} <= set(d)
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"]) and d["roofline"]["bound"] == "tensor"
    assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["d2h_bytes_per_step"] == 4 * 256 ** 3
    assert d["gpu_launches"] == 2 * d["steps"] and d["n_gpus"] == 1 and d["scaling"] == "weak"


def _last_line(name):
    with open(os.path.join(ROOT, "profiles", name)) as f:
        return json.loads([ln for ln in f if ln.startswith("{")][-1])


def test_round2_lines_have_the_contract_keys():
    """The committed round-2 lines (profiles/r2_bench_n1.json, r2_bench_n8.json): base contract, the tier's roofline /
    cpu_baseline / e2e objects, and the things VERDICT r1 asked to see in the driver record - the in-tolerance precision with
    its accuracy measured in the run, and at N > 1 the sharded 512^3 decode as the headline with its bit-identity flag."""
    d = _last_line("r2_bench_n1.json")
    assert BASE_KEYS <= set(d) and {"clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"} <= set(d)
    assert d["n_gpus"] == 1 and d["scaling"] == "weak" and d["dtype"] == "bf16" and d["gpu_launches"] == 2 * d["steps"]
    assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9 and d["roofline"]["traffic"] > 0
    assert d["second_precision"]["dtype"] == "fp16" and d["second_precision"]["ms_per_step"] > 0
    acc = d["accuracy"]
    assert acc["fp16"]["within_north_star_2e-3"] is True and acc["fp16"]["max_abs_vs_fp32"] < 2e-3
    assert acc["bf16"]["sign_agreement_where_abs_gt_2e-3"] >= 0.999 and acc["fp16"]["sign_agreement_where_abs_gt_2e-3"] >= 0.999
    assert d["e2e"]["d2h_bytes_per_step"] == 4 * 256 ** 3 and d["e2e_pageable"]["same_bits_as_pinned"] is True
    assert d["sparse_extraction"]["identical_triangle_soup"] is True and d["sparse_extraction"]["local_slopes"]["identical_triangle_soup"] is True
    assert {"ddpm_train_step", "decoder_train_step"} <= set(d["training"])
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1

    m = _last_line("r2_bench_n8.json")
    assert BASE_KEYS <= set(m) and m["n_gpus"] == 8 and m["scaling"] == "strong"
    c5 = m["config5_512cubed_sharded"]
    assert c5["bit_identical"] is True and abs(m["ms_per_step"] - c5["ms_per_step"]) < 1e-9
    assert abs(m["value"] - 512 ** 3 / (c5["ms_per_step"] * 1e-3)) < 1e-3 * m["value"]
    assert c5["ms_per_step"] < 50 and c5["second_precision"]["dtype"] == "fp16" and c5["second_precision"]["ms_per_step"] < 50
    assert "512" in m["config"]["workload"] and m["e2e"]["d2h_bytes_per_step"] > 0


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(pkg, tmp_path):
    """--dump-outputs DIR: the seeded sample of the headline decode_grid(z, 256) written after --steps timed steps is the same
    on a second run with another step count, and is what the package's own decode of the benchmark's latent returns."""
    import torch
    import bench
    legs_off = ["--no-cpu-baseline", "--no-accuracy", "--no-second-precision", "--no-config4", "--no-ddpm", "--no-vjp", "--no-train"]
    dumped = []
    for steps in (2, 3):
        out_dir = tmp_path / f"steps{steps}"
        proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                               "--dump-outputs", str(out_dir), *legs_off], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert proc.returncode == 0, proc.stderr[-2000:]
        lines = [ln for ln in proc.stdout.splitlines() if ln.strip()]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
        assert sorted(os.listdir(out_dir)) == ["sdf.npy"]
        assert sum(os.path.getsize(out_dir / f) for f in os.listdir(out_dir)) <= 64_000_000
        dumped.append(np.load(out_dir / "sdf.npy"))
    assert dumped[0].dtype == np.float32 and dumped[0].size > 3_000_000
    assert np.array_equal(dumped[0], dumped[1])
    dec = pkg.Decoder(pkg.synthetic.decoder_params(), device="cuda:0", precision="bf16")
    sdf = dec.decode_grid(torch.from_numpy(pkg.synthetic.latent(0)).cuda(), 256)
    assert np.array_equal(dumped[0], bench.dump_sample(sdf, 0))
    dec.close()
