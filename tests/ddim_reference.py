"""CPU reference of respaced (DDIM) sampling and deterministic DDIM inversion on the latent DDPM's
1000-step linear-beta schedule.  Test infrastructure only, like ``oracle/``, whose denoisers it reuses.

Op order (the C ABI's sdfb_ddim_schedule, the fused kernel's epilogue and the FFMA update follow it):
  x0 = clamp(sra x - srm1 eps, -clamp, clamp);  x <- c1 x0 + c2 x [+ c3 eps] [+ sigma z]
each product and sum rounded on its own, the c3 term only when c3 != 0, the noise term only when sigma != 0.
Coefficients are computed in fp64 and cast to fp32, like ``oracle.ddpm_schedule``.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from oracle import denoiser_forward, denoiser_forward_lowp
from oracle.weights import DDPM_T, DDPM_LATENT


def _abar():
    beta = np.linspace(1e-4, 0.02, DDPM_T, dtype=np.float64)
    return np.cumprod(1.0 - beta)


def ddim_timesteps(S: int) -> np.ndarray:
    """tau_i = floor(i T / S), i = 0 .. S-1 (the identity at S = T)."""
    return np.array([i * DDPM_T // S for i in range(S)], dtype=np.int64)


def ddim_schedule(S: int, eta: float, inverse: bool = False):
    """(timesteps int32 [S], rows float32 [S, 8]) in execution order; a row is
    (sra, srm1, c1, c2, c3, sigma, clamp, 0)."""
    ts, rows = _schedule_f64(S, eta, inverse)
    return ts, rows.astype(np.float32)


def _schedule_f64(S: int, eta: float, inverse: bool):
    if not 1 <= S <= DDPM_T:
        raise ValueError("1 <= S <= 1000")
    eta = float(np.float32(eta))          # the C ABI takes eta as a float
    if not 0.0 <= eta <= 1.0:
        raise ValueError("0 <= eta <= 1")
    ab = _abar()
    tau = ddim_timesteps(S)
    order = range(S) if inverse else range(S - 1, -1, -1)
    ts, rows = [], []
    for i in order:
        ts.append(tau[i])
        if inverse:
            cur = float(ab[tau[i - 1]]) if i > 0 else 1.0
            nxt = float(ab[tau[i]])
            rows.append([1.0 / math.sqrt(cur), math.sqrt(1.0 / cur - 1.0), math.sqrt(nxt), 0.0, math.sqrt(1.0 - nxt), 0.0,
                         math.inf, 0.0])
        else:
            a = float(ab[tau[i]])
            ap = float(ab[tau[i - 1]]) if i > 0 else 1.0
            sigma = eta * math.sqrt((1.0 - ap) / (1.0 - a)) * math.sqrt(1.0 - a / ap)
            c2 = math.sqrt(max(0.0, 1.0 - ap - sigma * sigma)) / math.sqrt(1.0 - a)
            c1 = math.sqrt(ap) - c2 * math.sqrt(a)
            rows.append([1.0 / math.sqrt(a), math.sqrt(1.0 / a - 1.0), c1, c2, 0.0, sigma, 1.0, 0.0])
    return np.array(ts, dtype=np.int32), np.array(rows, dtype=np.float64)


def ddim_update(x, eps, z, row, dtype):
    """One step of the respaced update, op for op (``row`` = 8 fp64 coefficients, cast to ``dtype``: fp32 gives the
    rows of ``ddim_schedule``, fp64 keeps them exact)."""
    c = [torch.tensor(float(v), dtype=dtype) for v in row[:7]]
    sra, srm1, c1, c2, c3, sigma, clamp = c
    x0 = torch.clamp(sra * x - srm1 * eps, -clamp, clamp)
    out = c1 * x0 + c2 * x
    if float(row[4]) != 0.0:
        out = out + c3 * eps
    if float(row[5]) != 0.0:
        out = out + sigma * z
    return out


def _eps(x, t, params, dtype, lowp):
    if lowp is None:
        return denoiser_forward(x, int(t), params=params, dtype=dtype)
    return denoiser_forward_lowp(x, int(t), params=params, lowp=lowp).to(dtype)


def _run(x, ts, rows, noise, S, params, dtype, lowp, inverse):
    nz = None if noise is None else torch.as_tensor(np.asarray(noise), dtype=dtype)
    for k in range(S):
        plane = k if inverse else S - 1 - k
        eps = _eps(x, ts[k], params, dtype, lowp)
        z = nz[plane] if (nz is not None and float(rows[k][5]) != 0.0) else None
        x = ddim_update(x, eps, z, rows[k], dtype)
    return x.numpy()


def ddim_sample(n: int, x_T, noise, S: int, eta: float, params=None, dtype=torch.float32, lowp=None):
    """DDIM from x_T [n,256] over S respaced steps; ``noise`` [S, n, 256] (noise[i] consumed at the step from tau_i;
    may be None when eta = 0).  ``lowp`` selects the tensor-core-emulating denoiser."""
    ts, rows = _schedule_f64(S, eta, False)
    x = torch.as_tensor(np.asarray(x_T), dtype=dtype).reshape(n, DDPM_LATENT).clone()
    return _run(x, ts, rows, noise, S, params, dtype, lowp, inverse=False)


def ddim_invert(x0, S: int, params=None, dtype=torch.float32, lowp=None):
    """Deterministic DDIM inversion of clean latents x0 [n,256] to x at tau_{S-1} (x0-hat is not clamped)."""
    ts, rows = _schedule_f64(S, 0.0, True)
    x = torch.as_tensor(np.asarray(x0), dtype=dtype).reshape(-1, DDPM_LATENT).clone()
    return _run(x, ts, rows, None, S, params, dtype, lowp, inverse=True)


def constant_eps_params(c: float = 0.125):
    """A denoiser whose weights are all zero and whose output bias is ``c``: eps_hat = c everywhere, at every t."""
    from oracle.weights import DDPM_LAYER_DIMS
    params = []
    for fin, fout in DDPM_LAYER_DIMS:
        params.append((np.zeros((fout, fin), np.float32), np.zeros(fout, np.float32)))
    params[-1] = (params[-1][0], np.full(params[-1][1].shape, c, np.float32))
    return params
