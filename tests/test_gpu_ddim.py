"""GPU tests of respaced (DDIM) sampling and DDIM inversion: the FFMA path against the fp32 reference (1e-4), the fused
tensor-core sampler against the reference that emulates its operand rounding, seeded against explicit noise bit for
bit, the full-length eta = 1 schedule against the DDPM sampler, and an exact round trip through a constant-noise
denoiser that pins the table wiring independently of the network."""
import numpy as np
import pytest
import torch

import oracle
from ddim_reference import constant_eps_params, ddim_invert, ddim_sample, ddim_schedule, ddim_timesteps

pytestmark = pytest.mark.gpu

LOWP_T = {"bf16": torch.bfloat16, "fp16": torch.float16}


def _stats(d):
    d = np.abs(d).ravel()
    q = np.quantile(d, [0.5, 0.9, 0.99])
    return f"p50 {q[0]:.2e} p90 {q[1]:.2e} p99 {q[2]:.2e} max {d.max():.2e}", q, d.max()


def _inputs(n, S, seed):
    rs = np.random.RandomState(seed)
    return rs.standard_normal((n, 256)).astype(np.float32), rs.standard_normal((S, n, 256)).astype(np.float32)


@pytest.mark.parametrize("S,eta", [(10, 0.0), (10, 1.0), (50, 0.0), (50, 1.0)])
def test_ddim_fp32_matches_reference(cuda_ddpm, S, eta):
    n = 5
    x_T, noise = _inputs(n, S, S)
    x = cuda_ddpm.sample_latents_ddim(n, steps=S, eta=eta, x_T=x_T, noise=noise, precision="fp32").cpu().numpy()
    ref = ddim_sample(n, x_T, noise, S, eta)
    err = np.abs(x - ref).max()
    print(f"ddim fp32 S={S} eta={eta}: max|kernel - reference| = {err:.2e}")
    assert err < 1e-4 and np.abs(x).max() <= 1.0 + 1e-6
    if eta == 0:      # no noise is read at eta = 0
        x2 = cuda_ddpm.sample_latents_ddim(n, steps=S, eta=eta, x_T=x_T, precision="fp32").cpu().numpy()
        assert np.array_equal(x, x2)


def test_ddim_inversion_fp32_matches_reference(cuda_ddpm):
    S, n = 50, 5
    x0 = (np.random.RandomState(1).standard_normal((n, 256)) * 0.5).astype(np.float32)
    x = cuda_ddpm.invert_latents_ddim(x0, steps=S, precision="fp32").cpu().numpy()
    ref = ddim_invert(x0, S)
    err = np.abs(x - ref).max()
    print(f"ddim inversion fp32 S={S}: max|kernel - reference| = {err:.2e} (|x_T| max {np.abs(ref).max():.2f})")
    assert err < 1e-4 * max(1.0, float(np.abs(ref).max()))


# Tile modes as the DDPM tests force them with SDFB_DDPM_BN (0 = automatic): 1100 runs 128-wide tiles in 16-CTA clusters,
# 3000 picks 256-wide tiles, 5000 puts two tiles on some pairs.
#
# Bounds.  Kernel and reference differ only in fp32 summation order, which matters where it flips a 16-bit rounding of a
# hidden activation: one evaluation of eps_hat differs by up to TOL_EPS_MAX (the bound of the DDPM single-step tests).
# A step passes an eps_hat difference into x with a gain of |c1 srm1 - c3| - up to 1.4 at S = 10 and 3.9 at S = 4 against
# at most 0.02 for a DDPM step - so the truncated DDPM runs' max bounds do not carry over.  The max bound here is the
# first-order one, TOL_EPS_MAX times the schedule's summed gain.  p90, which a wrong schedule row (timestep, coefficient
# or noise plane) breaks for every latent, keeps the DDPM runs' bound for bf16.
TOL_EPS_MAX = {"bf16": 2e-2, "fp16": 3e-3}
TOL_P90 = {"bf16": 2e-3, "fp16": 1e-3}


def _summed_gain(S, eta, inverse):
    _, rows = ddim_schedule(S, eta, inverse=inverse)
    r = rows.astype(np.float64)
    return float(np.abs(r[:, 2] * r[:, 1] - r[:, 4]).sum())


@pytest.mark.parametrize("mode", ["eta0", "eta1", "invert"])
@pytest.mark.parametrize("prec,n,bn,S", [("bf16", 37, 0, 10), ("bf16", 515, 0, 8), ("bf16", 515, 64, 8), ("bf16", 1100, 128, 6),
                                         ("bf16", 3000, 0, 4), ("bf16", 5000, 256, 4), ("fp16", 37, 0, 10), ("fp16", 1100, 0, 6)])
def test_ddim_tensor_core_matches_lowp_reference(cuda_ddpm, monkeypatch, prec, n, bn, S, mode):
    if bn:
        monkeypatch.setenv("SDFB_DDPM_BN", str(bn))
    x_T, noise = _inputs(n, S, n + S)
    if mode == "invert":
        x0 = (x_T * 0.5).astype(np.float32)
        run = lambda: cuda_ddpm.invert_latents_ddim(x0, steps=S, precision=prec)
        ref = ddim_invert(x0, S, lowp=LOWP_T[prec])
    else:
        eta = 0.0 if mode == "eta0" else 1.0
        run = lambda: cuda_ddpm.sample_latents_ddim(n, steps=S, eta=eta, x_T=x_T, noise=noise, precision=prec)
        ref = ddim_sample(n, x_T, noise, S, eta, lowp=LOWP_T[prec])
    x = run().cpu().numpy()
    msg, q, mx = _stats(x - ref)
    scale = max(1.0, float(np.abs(ref).max()))
    print(f"{prec} ddim {mode} n={n} bn={bn} S={S}: |kernel - {prec} reference| {msg} (|ref| max {scale:.2f})")
    assert np.isfinite(x).all()
    gain = _summed_gain(S, 0.0 if mode != "eta1" else 1.0, mode == "invert")
    assert mx < TOL_EPS_MAX[prec] * gain * scale, gain
    assert q[1] < TOL_P90[prec] * scale
    assert np.array_equal(x, run().cpu().numpy())        # deterministic


def test_seeded_ddim_equals_explicit_stream(cuda_ddpm, pkg, monkeypatch):
    """In-kernel noise (Philox step field tau_i, x_T from row 1000) == the same stream passed explicitly, bit for bit,
    on the fused kernel and on the FFMA path."""
    monkeypatch.setenv("SDFB_DDPM_BN", "256")
    n, S, seed = 300, 20, 2024
    tau = ddim_timesteps(S)
    noise = torch.stack([pkg.philox_normal(seed, n, int(t), int(t) + 1)[0] for t in tau])
    x_T = pkg.philox_normal(seed, n, 1000, 1001)[0]
    for prec in ("bf16", "fp32"):
        a = cuda_ddpm.sample_latents_ddim(n, steps=S, eta=1.0, seed=seed, precision=prec)
        b = cuda_ddpm.sample_latents_ddim(n, steps=S, eta=1.0, x_T=x_T, seed=seed, precision=prec)
        c = cuda_ddpm.sample_latents_ddim(n, steps=S, eta=1.0, x_T=x_T, noise=noise, precision=prec)
        assert torch.equal(a, b) and torch.equal(a, c), prec
        a0 = cuda_ddpm.sample_latents_ddim(n, steps=S, eta=0.0, seed=seed, precision=prec)
        c0 = cuda_ddpm.sample_latents_ddim(n, steps=S, eta=0.0, x_T=x_T, precision=prec)
        assert torch.equal(a0, c0) and not torch.equal(a0, a), prec


def test_seeded_ddim_is_addressed_by_global_latent_index(cuda_ddpm, monkeypatch):
    monkeypatch.setenv("SDFB_DDPM_BN", "128")
    n, S, seed = 600, 15, 99
    for prec in ("bf16", "fp32"):
        whole = cuda_ddpm.sample_latents_ddim(n, steps=S, eta=1.0, seed=seed, precision=prec)
        a = cuda_ddpm.sample_latents_ddim(256, steps=S, eta=1.0, seed=seed, precision=prec, first_latent=0)
        b = cuda_ddpm.sample_latents_ddim(n - 256, steps=S, eta=1.0, seed=seed, precision=prec, first_latent=256)
        assert torch.equal(torch.cat([a, b]), whole), prec


def test_ddim_batch_split_over_two_concurrent_launches(cuda_ddpm, monkeypatch):
    """4096 latents: both launches of the split read the one schedule table (see the DDPM test of the same name)."""
    S, seed = 25, 5
    whole = cuda_ddpm.sample_latents_ddim(4096, steps=S, eta=1.0, seed=seed, precision="bf16")
    ms = cuda_ddpm.last_kernel_ms()
    a = cuda_ddpm.sample_latents_ddim(3840, steps=S, eta=1.0, seed=seed, precision="bf16", first_latent=0)
    monkeypatch.setenv("SDFB_DDPM_BN", "128")
    b128 = cuda_ddpm.sample_latents_ddim(256, steps=S, eta=1.0, seed=seed, precision="bf16", first_latent=3840)
    monkeypatch.setenv("SDFB_DDPM_BN", "256")
    b256 = cuda_ddpm.sample_latents_ddim(256, steps=S, eta=1.0, seed=seed, precision="bf16", first_latent=3840)
    split = torch.equal(whole[3840:], b128)
    print(f"ddim 4096 latents x {S} steps: {ms * 1e3 / S:.1f} us/step ({'15 clusters + plain pairs' if split else '16 clusters'})")
    assert torch.equal(whole[:3840], a)
    assert split or torch.equal(whole[3840:], b256)


def test_full_length_eta_one_ddim_is_the_ddpm_chain(cuda_ddpm):
    n, seed = 8, 77
    for prec, tol in (("fp32", 1e-4), ("bf16", 3e-2)):
        ddpm = cuda_ddpm.sample_latents(n, seed=seed, precision=prec).cpu().numpy()
        ddim = cuda_ddpm.sample_latents_ddim(n, steps=1000, eta=1.0, seed=seed, precision=prec).cpu().numpy()
        err = np.abs(ddim - ddpm).max()
        print(f"{prec}: max|DDIM(S=1000, eta=1) - DDPM| = {err:.2e}")
        assert err < tol


@pytest.fixture(scope="module")
def constant_eps_ddpm(pkg):
    m = pkg.LatentDDPM(oracle.flatten_params(constant_eps_params()), device="cuda:0", precision="fp32")
    yield m
    m.close()


@pytest.mark.parametrize("prec", ["fp32", "bf16", "fp16"])
def test_round_trip_through_a_constant_noise_prediction(constant_eps_ddpm, prec):
    """eps_hat is exactly the same constant on every path (zero weights), so inversion followed by eta = 0 sampling
    must return x0 up to fp32 rounding, and every precision must compute the fp32 reference's numbers."""
    S, n = 50, 515
    params = constant_eps_params()
    x0 = np.random.RandomState(4).uniform(-0.5, 0.5, (n, 256)).astype(np.float32)
    x_T = constant_eps_ddpm.invert_latents_ddim(x0, steps=S, precision=prec)
    back = constant_eps_ddpm.sample_latents_ddim(n, steps=S, eta=0.0, x_T=x_T, precision=prec).cpu().numpy()
    ref_T = ddim_invert(x0, S, params=params)
    ref = ddim_sample(n, ref_T, None, S, 0.0, params=params)
    err, dref = np.abs(back - x0).max(), np.abs(back - ref).max()
    print(f"{prec} constant-eps round trip S={S}: max|back - x0| = {err:.2e}, max|back - fp32 reference| = {dref:.2e}")
    assert np.abs(x_T.cpu().numpy() - ref_T).max() < 1e-5
    assert err < 1e-4 and dref < 1e-5
