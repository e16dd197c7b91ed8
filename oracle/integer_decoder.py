"""An integer-valued decoder network and its exact reference (test infrastructure only).

Every value the decoder adds up - in the fp32 FFMA chain, in the tensor core's fp32 accumulator, in the
latent fold - is an integer (the head's terms: a multiple of 2^-8), and every partial sum stays below 2^24
of those units.  Then:

  * every fp32 sum is exact in any order, so there is no summation-order noise between two correct
    implementations;
  * every 16-bit rounding of an integer >= 1 gives an integer again (round to nearest even, deterministic)
    and a positive integer never rounds to 0;

so the decoder's pre-activation x = h7 . w8 + b8 has exactly one correct value at every query, in every tile
and at every precision, and a kernel can be compared with it exactly instead of by tolerance.

The construction (parameters in the C-ABI layout of ``oracle.weights``, seeded by ``numpy.random.RandomState``):

  * layer 0: the xyz columns of W0 are 256 times small integers.  A grid coordinate of res = 2^k + 1 (rule A1)
    is j / 2^(k-1), a dyadic point j / 256, so W0x . xyz is an integer for every res <= 513; the latent
    columns of W0 and W4 are sparse ternary {-1, 0, 1} and latents are small integers, so the folded biases
    bias0' = b0 + W0z z and bias4' = b4 + W4z z are integers;
  * layers 1..7: sparse ternary weights (``NNZ`` nonzeros per row), integer biases;
  * layer 4: the xyz columns are 256 times small integers; j / 256 with |j| <= 256 is exact in bf16 and fp16,
    so the 16-bit rounding of the coordinates that ride in layer 3's padding columns changes nothing;
  * head: w8 and b8 are multiples of 2^-8.

``forward`` does not take this on trust: next to every layer it evaluates |a| @ |W|^T + |b| (the largest
partial sum any summation order can meet) at every query it evaluates and checks it against 2^24 units, and
with fp16 it checks that no activation overflows.
"""
from __future__ import annotations

from functools import lru_cache

import numpy as np
import torch

from .weights import DEC_HIDDEN, DEC_LATENT, DEC_LAYER_DIMS, DEC_SKIP_OUT

INT_WEIGHT_SEED = 17
INT_LATENT_SEED = 23
NNZ = 3                       # nonzeros per row of the ternary hidden layers
HEAD_WINDOW = 32              # layer 7 comes in unit pairs relu(u + b) - relu(u + b - HEAD_WINDOW): u clamped to a window
HEAD_UNIT = 2.0 ** -8         # granule of the head's terms (w8, b8 and h7 . w8)
EXACT_LIMIT = 2.0 ** 24       # a sum of integers below this (in its own units) is exact in fp32
FP16_MAX = 65504.0
# Chosen once as minus the median of h7 . w8 over the 129^3 grid at latent 1 (a value that product takes), so that
# about half of every grid is inside and that latent's field has exact zeros.
INT_HEAD_BIAS = -0.125

LOWP = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": None}


def _ternary_rows(rs, fout, fin, nnz):
    w = np.zeros((fout, fin))
    for n in range(fout):
        cols = rs.choice(fin, nnz, replace=False)
        w[n, cols] = rs.choice((-1.0, 1.0), nnz)
    return w


@lru_cache(maxsize=None)
def integer_decoder_weights():
    """List of (W[out,in] float32, b[out] float32) for the nine decoder layers, integer-valued as described above."""
    rs = np.random.RandomState(INT_WEIGHT_SEED)
    L, S = DEC_LATENT, DEC_SKIP_OUT
    params = []
    for li, (fin, fout) in enumerate(DEC_LAYER_DIMS):
        if li == 0:
            w = np.zeros((fout, fin))
            w[:, :L] = _ternary_rows(rs, fout, L, 3)
            w[:, L:] = 256.0 * rs.randint(-1, 2, size=(fout, 3))
            b = rs.randint(-160, 161, size=fout).astype(np.float64)
        elif li == 4:
            w = np.zeros((fout, fin))
            w[:, :S] = _ternary_rows(rs, fout, S, NNZ)
            w[:, S:S + L] = _ternary_rows(rs, fout, L, 3)
            w[:, S + L:] = 256.0 * rs.randint(-1, 2, size=(fout, 3))
            b = rs.randint(-8, 25, size=fout).astype(np.float64)
        elif li < 7:
            w = _ternary_rows(rs, fout, fin, NNZ)
            b = rs.randint(-8, 25, size=fout).astype(np.float64)
        elif li == 7:
            w = np.repeat(_ternary_rows(rs, fout // 2, fin, NNZ), 2, axis=0)
            b = np.repeat(rs.randint(-64, 65, size=fout // 2), 2).astype(np.float64)
            b[1::2] -= HEAD_WINDOW
        else:
            w = np.repeat(rs.choice((-1.0, 1.0), size=(fout, fin // 2)), 2, axis=1) * HEAD_UNIT
            w[:, 1::2] *= -1.0
            b = np.full(fout, INT_HEAD_BIAS)
        params.append((np.ascontiguousarray(w, dtype=np.float32), np.ascontiguousarray(b, dtype=np.float32)))
    return params


def integer_latent(index: int) -> np.ndarray:
    """Latent code [256] float32 of small integers in [-3, 3]; index 0 is the zero latent."""
    if index == 0:
        return np.zeros(DEC_LATENT, np.float32)
    rs = np.random.RandomState(INT_LATENT_SEED + 1000 * index)
    return rs.randint(-3, 4, size=DEC_LATENT).astype(np.float32)


def dyadic_points(m: int, seed: int = 0) -> np.ndarray:
    """[m, 3] float32 query points, random multiples of 1/256 in [-1, 1]."""
    rs = np.random.RandomState(seed)
    return (rs.randint(-256, 257, size=(m, 3)) / 256.0).astype(np.float32)


def grid_xyz(res: int, q0: int, q1: int, device=None) -> torch.Tensor:
    """float64 [q1 - q0, 3] coordinates of grid queries [q0, q1) (x fastest; rule A1, exact for res = 2^k + 1)."""
    q = torch.arange(q0, q1, dtype=torch.int64, device=device)
    ix, iy, iz = q % res, (q // res) % res, q // (res * res)
    num = torch.stack([ix, iy, iz], dim=1) * 2 - (res - 1)
    return num.to(torch.float64) / (res - 1)


class PremiseError(AssertionError):
    pass


class Stats:
    """What ``forward`` saw, accumulated over chunks: the largest premise bound per layer (in units of the layer's
    term granule), the largest activation before a 16-bit rounding, and per-layer activity counts."""

    def __init__(self):
        self.bound = [0.0] * 9
        self.max_act = 0.0
        self.queries = 0
        self.active_units = [0] * 8        # sum over queries of the number of positive pre-activations
        self.dead_queries = [0] * 8        # queries at which a layer has no positive pre-activation at all

    def merge(self, other: "Stats"):
        self.bound = [max(a, b) for a, b in zip(self.bound, other.bound)]
        self.max_act = max(self.max_act, other.max_act)
        self.queries += other.queries
        self.active_units = [a + b for a, b in zip(self.active_units, other.active_units)]
        self.dead_queries = [a + b for a, b in zip(self.dead_queries, other.dead_queries)]

    def active_fraction(self, layer: int) -> float:
        width = DEC_SKIP_OUT if layer == 3 else DEC_HIDDEN
        return self.active_units[layer] / max(self.queries * width, 1)

    def summary(self) -> str:
        b = ", ".join(f"L{i} {v:.0f}" for i, v in enumerate(self.bound))
        a = ", ".join(f"{self.active_fraction(i):.2f}" for i in range(8))
        return f"premise bound per layer (limit 2^24 = {EXACT_LIMIT:.0f}): {b}; active fraction h0..h7: {a}; " \
               f"largest activation {self.max_act:.0f}"


def _t(a, device):
    return torch.as_tensor(np.asarray(a), dtype=torch.float64, device=device)


@lru_cache(maxsize=16)
def _layers(device_str: str, lowp_name: str):
    """float64 weights (16-bit rounded where the kernel rounds them) and their absolute values, on a device."""
    dev = torch.device(device_str)
    lowp = LOWP[lowp_name]
    P = integer_decoder_weights()
    L, S = DEC_LATENT, DEC_SKIP_OUT
    rnd = (lambda t: t) if lowp is None else (lambda t: t.to(torch.float32).to(lowp).to(torch.float64))
    W = [_t(w, dev) for w, _ in P]
    B = [_t(b, dev) for _, b in P]
    lay = {"W0z": W[0][:, :L], "W0x": W[0][:, L:], "b0": B[0], "W4z": W[4][:, S:S + L], "b4": B[4],
           "W4": torch.cat([rnd(W[4][:, :S]), rnd(W[4][:, S + L:])], dim=1),
           "w8": W[8][0], "b8": B[8]}
    for i in (1, 2, 3, 5, 6, 7):
        lay[f"W{i}"], lay[f"b{i}"] = rnd(W[i]), B[i]
    # one product per layer gives the value and the bound: a @ [W ; |W|]^T
    for i in range(1, 8):
        Wi = lay[f"W{i}"]
        lay[f"WW{i}"] = torch.cat([Wi, Wi.abs()], dim=0).T.contiguous()
    return lay


def forward(latent, xyz, lowp: str = "bf16", preacts: bool = False, stats: Stats | None = None):
    """The decoder's data path in float64 (exact on this network), on xyz's device.

    ``lowp``: "bf16" / "fp16" emulate the tensor-core kernel (oracle.decoder_forward_lowp: activations h0..h6,
    the hidden weights and layer 4's coordinates rounded to 16 bits, h7 and the head unrounded); "fp32" is the
    FFMA path (no rounding).  ``xyz``: float64 tensor [m, 3] (or anything torch.as_tensor takes).
    Returns x = h7 . w8 + b8 [m] float64 and, with ``preacts``, the pre-activations of layers 0..7 ([m, 512],
    layer 3: [m, 253]).  Raises PremiseError where the exactness premise fails; ``stats`` accumulates what was seen.
    """
    xyz = torch.as_tensor(xyz, dtype=torch.float64)
    dev = xyz.device
    lay = _layers(str(dev), lowp)
    lp = LOWP[lowp]
    rnd = (lambda t: t) if lp is None else (lambda t: t.to(torch.float32).to(lp).to(torch.float64))
    z = _t(latent, dev).reshape(DEC_LATENT)
    st = Stats()
    st.queries = xyz.shape[0]

    def check(layer, bound, unit=1.0):
        m = float(bound.max()) / unit if bound.numel() else 0.0
        st.bound[layer] = max(st.bound[layer], m)
        if not m < EXACT_LIMIT:
            raise PremiseError(f"layer {layer}: a partial sum may reach {m:.0f} units of {unit}: not exact in fp32")

    def act(layer, pre, rounded):
        pos = pre > 0
        st.active_units[layer] += int(pos.sum())
        st.dead_queries[layer] += int((~pos.any(dim=1)).sum())
        h = torch.relu(pre)
        if rounded:
            st.max_act = max(st.max_act, float(h.max()) if h.numel() else 0.0)
            if lp == torch.float16 and not st.max_act < FP16_MAX:
                raise PremiseError(f"layer {layer}: activation {st.max_act:.0f} overflows fp16")
            h = rnd(h)
        return h

    pre = []
    bias0 = lay["b0"] + lay["W0z"] @ z
    bias0_bound = lay["b0"].abs() + lay["W0z"].abs() @ z.abs()
    p = xyz @ lay["W0x"].T + bias0
    check(0, xyz.abs() @ lay["W0x"].abs().T + bias0_bound)
    pre.append(p)
    h = act(0, p, True)
    for i in range(1, 8):
        if i == 4:
            S = DEC_SKIP_OUT
            a = torch.cat([h, rnd(xyz)], dim=1)
            W4 = lay["W4"]
            bias4 = lay["b4"] + lay["W4z"] @ z
            p = a @ W4.T + bias4
            check(4, a.abs() @ W4.abs().T + lay["b4"].abs() + lay["W4z"].abs() @ z.abs())
        else:
            vb = h @ lay[f"WW{i}"]
            n = vb.shape[1] // 2
            p = vb[:, :n] + lay[f"b{i}"]
            check(i, vb[:, n:] + lay[f"b{i}"].abs())
        pre.append(p)
        h = act(i, p, i < 7)
    x = h @ lay["w8"] + lay["b8"][0]
    check(8, h @ lay["w8"].abs() + lay["b8"][0].abs(), HEAD_UNIT)
    if stats is not None:
        stats.merge(st)
    return (x, pre) if preacts else x


def forward_grid(latent, res: int, lowp: str = "bf16", q0: int = 0, q1: int | None = None, device=None,
                 chunk: int = 1 << 16, stats: Stats | None = None) -> torch.Tensor:
    """x [q1 - q0] float64 of grid queries [q0, q1) of the res^3 grid, evaluated in chunks on ``device``."""
    q1 = res ** 3 if q1 is None else q1
    out = torch.empty(q1 - q0, dtype=torch.float64, device=device)
    for s in range(q0, q1, chunk):
        e = min(q1, s + chunk)
        out[s - q0:e - q0] = forward(latent, grid_xyz(res, s, e, device), lowp, stats=stats)
    return out


def forward_points(latent, xyz, lowp: str = "bf16", device=None, chunk: int = 1 << 16,
                   stats: Stats | None = None) -> torch.Tensor:
    """x [m] float64 of query points xyz [m, 3], evaluated in chunks on ``device``."""
    pts = torch.as_tensor(np.asarray(xyz), dtype=torch.float64).reshape(-1, 3)
    out = torch.empty(pts.shape[0], dtype=torch.float64, device=device)
    for s in range(0, pts.shape[0], chunk):
        e = min(pts.shape[0], s + chunk)
        out[s:e] = forward(latent, pts[s:e].to(device), lowp, stats=stats)
    return out
