"""CPU tests of the drop-in boundary: the C-ABI library loads and exports every symbol
include/sdfb200.h declares, and refuses to run without a device (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "sdfb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sdfb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(pkg):
    lib = pkg.load_library()
    names = declared_symbols()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"libsdfb200.so does not export {n}"
    from importlib import import_module
    sigs = import_module(pkg.__name__ + "._lib").SIGNATURES
    assert sorted(sigs) == names, "ctypes signature table and header disagree"
    assert lib.sdfb_version() >= 100


def test_header_constants_match_oracle(pkg):
    import oracle
    text = open(os.path.join(ROOT, "include", "sdfb200.h")).read()
    dec = int(re.search(r"SDFB_DECODER_PARAM_FLOATS (\d+)", text).group(1))
    ddp = int(re.search(r"SDFB_DDPM_PARAM_FLOATS (\d+)", text).group(1))
    assert dec == oracle.flatten_params(oracle.decoder_weights()).size
    assert ddp == oracle.flatten_params(oracle.ddpm_weights()).size


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device error path")
def test_no_cpu_fallback(pkg):
    import oracle
    lib = pkg.load_library()
    flat = oracle.flatten_params(oracle.decoder_weights())
    h = C.c_void_p()
    rc = lib.sdfb_decoder_create(flat.ctypes.data, flat.size, 0, C.byref(h))
    assert rc == -2 and not h.value                      # SDFB_E_DEVICE
    assert b"no CPU path" in lib.sdfb_last_error() or b"device" in lib.sdfb_last_error()
    with pytest.raises(Exception):
        pkg.Decoder(flat, device="cuda:0")
    with pytest.raises(ValueError):
        pkg.Decoder(flat, device="cpu")


def test_argument_validation_without_device(pkg):
    lib = pkg.load_library()
    h = C.c_void_p()
    bad = np.zeros(10, np.float32)
    assert lib.sdfb_decoder_create(bad.ctypes.data, bad.size, 0, C.byref(h)) == -1   # wrong blob size
    assert lib.sdfb_decoder_create(None, 0, 0, C.byref(h)) == -1
    assert lib.sdfb_ddpm_create(bad.ctypes.data, bad.size, 0, C.byref(h)) == -1
    assert lib.sdfb_decoder_destroy(None) == 0
    assert lib.sdfb_ddpm_destroy(None) == 0


def test_workspace_queries_and_validation_of_the_extraction_entry_points(pkg):
    """Size queries need no device; bad shapes / null pointers are refused before anything is launched."""
    lib = pkg.load_library()
    b = C.c_size_t()
    assert lib.sdfb_mc_workspace_bytes(64, 64, 64, C.byref(b)) == 0 and b.value >= 64 ** 3 // 8
    assert lib.sdfb_mc_workspace_bytes(1, 64, 64, C.byref(b)) == -1
    n = C.c_int64()
    assert lib.sdfb_mc_count(None, None, 4, 4, 4, None, 0, C.byref(n), None) == -1
    assert lib.sdfb_decoder_vjp_latent(None, None, None, 0, None, None, None, None) == -1
    assert lib.sdfb_philox_normal(1, -1, 4, 0, 1, None, None) == -1
    assert lib.sdfb_ddpm_sample_philox(None, None, 0, 0, 4, 10, 1, 1, None) == -1


def test_header_is_valid_c_and_links_from_a_c_program(pkg, tmp_path):
    """include/sdfb200.h compiled as C99 with -Wall -Werror, linked against libsdfb200.so, run without a device."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not found")
    lib = os.path.join(ROOT, "latent-diffusion-models-for-shape-sdfs_b200", "libsdfb200.so")
    exe = str(tmp_path / "abi_smoke")
    cmd = [gcc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "c", "abi_smoke.c"), "-o", exe, lib, "-Wl,-rpath," + os.path.dirname(lib)]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    assert proc.returncode == 0, proc.stderr
    run = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert run.returncode == 0, (run.returncode, run.stdout, run.stderr)
    assert "sdfb C ABI ok" in run.stdout
