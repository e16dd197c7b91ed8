"""Host-side API: thin, validating wrappers that hand device pointers to the C ABI.

Names and argument meaning follow the oracle modules (oracle/decoder.py, oracle/ddpm.py),
which restate the method in SURVEY.md section 8(a); results are torch CUDA tensors.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import PRECISIONS, check

LATENT = 256
DDPM_STEPS = 1000
# The DDPM works on latents normalised to unit scale; a decoder latent is a sample times this (the N(0, 1/16^2) code scale
# of the auto-decoder, oracle/ddpm.py DDPM_LATENT_SCALE).  Unscaled samples (|x| up to 1 per component) saturate the decoder.
DDPM_LATENT_SCALE = 1.0 / 16.0


def _flat_params(params, expect: int) -> np.ndarray:
    """Accepts the flat blob (numpy / torch) or a list of (W[out,in], b[out]) pairs."""
    if isinstance(params, (list, tuple)):
        parts = []
        for w, b in params:
            parts.append(np.asarray(w, dtype=np.float32).ravel())
            parts.append(np.asarray(b, dtype=np.float32).ravel())
        flat = np.concatenate(parts)
    elif isinstance(params, torch.Tensor):
        flat = params.detach().cpu().numpy().astype(np.float32, copy=False).ravel()
    else:
        flat = np.asarray(params, dtype=np.float32).ravel()
    if flat.size != expect:
        raise ValueError(f"parameter blob has {flat.size} floats, expected {expect}")
    return np.ascontiguousarray(flat)


def _device_index(device) -> int:
    dev = torch.device(device)
    if dev.type != "cuda":
        raise ValueError("libsdfb200 runs on CUDA devices only (no CPU fallback)")
    return torch.cuda.current_device() if dev.index is None else dev.index


def _prec(precision: str) -> int:
    try:
        return PRECISIONS[precision]
    except KeyError:
        raise ValueError(f"precision must be one of {sorted(PRECISIONS)}, got {precision!r}") from None


def _stream_ptr(device_index: int) -> int:
    return torch.cuda.current_stream(device_index).cuda_stream


def _as_dev_f32(t, device: torch.device, shape=None) -> torch.Tensor:
    t = torch.as_tensor(np.asarray(t) if not isinstance(t, torch.Tensor) else t)
    t = t.to(device=device, dtype=torch.float32).contiguous()
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise ValueError(f"expected shape {tuple(shape)}, got {tuple(t.shape)}")
    return t


class Decoder:
    """DeepSDF-style auto-decoder (259 -> 512x3 -> 253 (+259 skip) -> 512x4 -> 1, tanh).

    ``Decoder(latent, xyz) -> sdf``; ``decode_grid(z, res)``.  ``precision``: "bf16" / "fp16"
    run the fused tcgen05 kernel, "fp32" the FFMA kernels.
    """

    def __init__(self, params, device="cuda:0", precision: str = "bf16"):
        self._lib = _lib.load()
        self.device = torch.device("cuda", _device_index(device))
        self.precision = precision
        _prec(precision)
        flat = _flat_params(params, _lib.DECODER_PARAM_FLOATS)
        handle = C.c_void_p()
        check(self._lib.sdfb_decoder_create(flat.ctypes.data, flat.size, self.device.index, C.byref(handle)))
        self._h = handle

    def close(self):
        if getattr(self, "_h", None):
            self._lib.sdfb_decoder_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- Decoder(latent, xyz) -> sdf ------------------------------------------------
    def __call__(self, latent, xyz, precision: str | None = None) -> torch.Tensor:
        prec = _prec(precision or self.precision)
        lat = _as_dev_f32(latent, self.device)
        pts = _as_dev_f32(xyz, self.device)
        if lat.ndim == 1:
            if lat.shape[0] != LATENT or pts.ndim != 2 or pts.shape[1] != 3:
                raise ValueError("expected latent [256] and xyz [M,3]")
            return self._points(lat, pts, prec)
        # batch of shapes: latent [B,256], xyz [B,M,3] -> sdf [B,M]
        if lat.ndim != 2 or lat.shape[1] != LATENT or pts.ndim != 3 or pts.shape[0] != lat.shape[0] or pts.shape[2] != 3:
            raise ValueError("expected latent [B,256] and xyz [B,M,3]")
        out = torch.empty(pts.shape[:2], dtype=torch.float32, device=self.device)
        for b in range(lat.shape[0]):
            out[b] = self._points(lat[b], pts[b], prec)
        return out

    def _points(self, lat, pts, prec) -> torch.Tensor:
        M = pts.shape[0]
        out = torch.empty(M, dtype=torch.float32, device=self.device)
        check(self._lib.sdfb_decode_points(self._h, lat.data_ptr(), pts.data_ptr() if M else None, M,
                                           out.data_ptr() if M else None, prec, _stream_ptr(self.device.index)))
        return out

    # ---- decode_grid(z, res) -> sdf[z,y,x] (+ mask) -------------------------------------
    def decode_grid(self, latent, res: int, z0: int = 0, z1: int | None = None, mask: bool = False,
                    precision: str | None = None, out: torch.Tensor | None = None):
        """sdf [z1-z0, res, res] float32 of planes [z0, z1); with ``mask=True`` also the uint8
        sign-change mask of cell layers [z0, min(z1, res-1)) as [layers, res-1, res-1].

        ``out`` (optional) is a preallocated float32 buffer; with ``mask`` and z1 < res it must
        hold one extra (halo) plane, which is decoded locally instead of being exchanged."""
        prec = _prec(precision or self.precision)
        z1 = res if z1 is None else z1
        if not (0 <= z0 <= z1 <= res) or res < 2:
            raise ValueError(f"bad plane range [{z0}, {z1}) for res {res}")
        lat = _as_dev_f32(latent, self.device, (LATENT,))
        halo = 1 if (mask and z1 < res and z1 > z0) else 0
        planes = z1 - z0 + halo
        if out is None:
            buf = torch.empty((planes, res, res), dtype=torch.float32, device=self.device)
        else:
            if out.dtype != torch.float32 or out.device != self.device or not out.is_contiguous() or out.numel() < planes * res * res:
                raise ValueError("out must be a contiguous float32 CUDA tensor with room for the slab (+ halo plane)")
            buf = out
        layers = (z1 if halo else min(z1, res - 1)) - z0
        m = None
        if mask:
            m = torch.empty((max(layers, 0), res - 1, res - 1), dtype=torch.uint8, device=self.device)
        if z1 == z0:            # an empty slab (tail rank of an uneven split): empty results, nothing launched
            sdf = buf.view(-1)[:0].view(0, res, res)
            return (sdf, m) if mask else sdf
        check(self._lib.sdfb_decode_grid(self._h, lat.data_ptr(), res, z0, z1, buf.data_ptr(),
                                         m.data_ptr() if (m is not None and m.numel()) else None, prec,
                                         _stream_ptr(self.device.index)))
        sdf = buf.view(-1)[: (z1 - z0) * res * res].view(z1 - z0, res, res)
        return (sdf, m) if mask else sdf

    def decode_grid_bits(self, latent, res: int, z0: int = 0, z1: int | None = None, mask: bool = True,
                         precision: str | None = None):
        """(sdf [z1-z0,res,res], sign_words int32 [ceil(M/32)], mask_words int32 [ceil(cells/32)] or None):
        the packed outputs - sign bit-planes written by the decoder kernel itself (bit q & 31 of word
        q >> 5, halo plane included) and the sign-change mask at one bit per cell."""
        prec = _prec(precision or self.precision)
        z1 = res if z1 is None else z1
        if not (0 <= z0 <= z1 <= res) or res < 2:
            raise ValueError(f"bad plane range [{z0}, {z1}) for res {res}")
        lat = _as_dev_f32(latent, self.device, (LATENT,))
        halo = 1 if (mask and z1 < res and z1 > z0) else 0
        planes = z1 - z0 + halo
        buf = torch.empty((planes, res, res), dtype=torch.float32, device=self.device)
        signs = torch.zeros(((planes * res * res + 31) // 32,), dtype=torch.int32, device=self.device)
        layers = (z1 if halo else min(z1, res - 1)) - z0
        cells = max(layers, 0) * (res - 1) * (res - 1)
        mw = torch.zeros(((cells + 31) // 32,), dtype=torch.int32, device=self.device) if mask else None
        check(self._lib.sdfb_decode_grid_bits(self._h, lat.data_ptr(), res, z0, z1, buf.data_ptr(),
                                              signs.data_ptr() if signs.numel() else None,
                                              mw.data_ptr() if (mw is not None and mw.numel()) else None, prec,
                                              _stream_ptr(self.device.index)))
        return buf[: z1 - z0], signs, mw

    # ---- gradient w.r.t. the latent (auto-decoder fitting) ----------------------------------------
    def latent_vjp(self, latent, xyz, dLdy, precision: str = "fp32"):
        """(grad [256], sdf [M]): grad = sum_m dLdy[m] * d sdf(latent, xyz_m) / d latent.
        ``precision="fp32"``: FFMA path; ``"bf16"`` / ``"fp16"``: one launch of the forward + backward instance of
        the fused tensor-core kernel (sdf is then what ``Decoder(latent, xyz)`` returns at that precision)."""
        prec = PRECISIONS[precision]
        lat = _as_dev_f32(latent, self.device, (LATENT,))
        pts = _as_dev_f32(xyz, self.device)
        up = _as_dev_f32(dLdy, self.device)
        if pts.ndim != 2 or pts.shape[1] != 3 or up.shape != (pts.shape[0],):
            raise ValueError("expected xyz [M,3] and dLdy [M]")
        M = pts.shape[0]
        grad = torch.empty(LATENT, dtype=torch.float32, device=self.device)
        sdf = torch.empty(M, dtype=torch.float32, device=self.device)
        if prec == PRECISIONS["fp32"]:
            check(self._lib.sdfb_decoder_vjp_latent(self._h, lat.data_ptr(), pts.data_ptr() if M else None, M,
                                                    up.data_ptr() if M else None, grad.data_ptr(),
                                                    sdf.data_ptr() if M else None, _stream_ptr(self.device.index)))
        else:
            check(self._lib.sdfb_decoder_vjp_latent_tc(self._h, lat.data_ptr(), pts.data_ptr() if M else None, M,
                                                       up.data_ptr() if M else None, grad.data_ptr(),
                                                       sdf.data_ptr() if M else None, prec,
                                                       _stream_ptr(self.device.index)))
        return grad, sdf

    def fit_loss_grad(self, latent, xyz, sdf_target, clamp: float = 0.1, precision: str = "bf16", return_sdf: bool = False):
        """(loss [1], grad [256]) of loss = mean |clamp(sdf(latent, xyz)) - clamp(sdf_target)| w.r.t. the latent, in ONE
        launch of the forward + backward instance of the fused kernel (the upstream gradient is formed in the kernel).
        Nothing is synchronised: both results stay on the device."""
        prec = PRECISIONS[precision]
        lat = _as_dev_f32(latent, self.device, (LATENT,))
        pts = _as_dev_f32(xyz, self.device)
        tgt = _as_dev_f32(sdf_target, self.device)
        if pts.ndim != 2 or pts.shape[1] != 3 or tgt.shape != (pts.shape[0],):
            raise ValueError("expected xyz [M,3] and sdf_target [M]")
        M = pts.shape[0]
        grad = torch.empty(LATENT, dtype=torch.float32, device=self.device)
        loss = torch.empty(1, dtype=torch.float32, device=self.device)
        sdf = torch.empty(M, dtype=torch.float32, device=self.device) if return_sdf else None
        check(self._lib.sdfb_decoder_fit_loss_grad(self._h, lat.data_ptr(), pts.data_ptr() if M else None, M,
                                                   tgt.data_ptr() if M else None, float(clamp), grad.data_ptr(),
                                                   loss.data_ptr(), sdf.data_ptr() if (sdf is not None and M) else None, prec,
                                                   _stream_ptr(self.device.index)))
        return (loss, grad, sdf) if return_sdf else (loss, grad)

    def fit_latent(self, xyz, sdf_target, steps: int = 300, lr: float = 5e-3, clamp: float = 0.1, reg: float = 1e-4,
                   init=None, precision: str = "fp32"):
        """Auto-decoder inference (DeepSDF's reconstruction step): Adam on the latent so that the decoded
        field matches ``sdf_target`` at ``xyz``; loss = mean |clamp(y) - clamp(s)| + reg |z|^2.
        ``precision``: arithmetic of the forward and backward passes ("bf16" / "fp16": tensor pipe).
        Returns (latent [256], last loss)."""
        pts = _as_dev_f32(xyz, self.device)
        tgt = torch.clamp(_as_dev_f32(sdf_target, self.device), -clamp, clamp)
        z = torch.zeros(LATENT, device=self.device) if init is None else _as_dev_f32(init, self.device, (LATENT,)).clone()
        m = torch.zeros_like(z)
        v = torch.zeros_like(z)
        M = pts.shape[0]
        if precision != "fp32":              # two launches per step (loss + gradient, Adam), nothing synchronised until the end
            loss_t = None
            st = _stream_ptr(self.device.index)
            for it in range(1, steps + 1):
                loss_t, g = self.fit_loss_grad(z, pts, tgt, clamp=clamp, precision=precision)
                # the loss reported belongs to the latent it was evaluated at: the kernel adds reg |z|^2 before it moves z
                check(self._lib.sdfb_latent_adam_step(z.data_ptr(), m.data_ptr(), v.data_ptr(), g.data_ptr(), loss_t.data_ptr(), 1,
                                                      float(lr), float(reg), 0.9, 0.999, 1e-8, it, st))
            loss = float(loss_t[0]) if loss_t is not None else float("nan")
            self.check()
            return z, loss
        ones = torch.ones(M, device=self.device)
        loss = float("nan")
        for it in range(1, steps + 1):
            if it == 1:
                y = self(z, pts, precision=precision)
            inside = (y > -clamp) & (y < clamp)
            dLdy = torch.sign(torch.clamp(y, -clamp, clamp) - tgt) * inside / M
            g, y_chk = self.latent_vjp(z, pts, dLdy, precision=precision)
            loss = float((torch.clamp(y_chk, -clamp, clamp) - tgt).abs().mean() + reg * (z * z).sum())
            g = g + 2 * reg * z
            m = 0.9 * m + 0.1 * g
            v = 0.999 * v + 0.001 * g * g
            z = z - lr * (m / (1 - 0.9 ** it)) / ((v / (1 - 0.999 ** it)).sqrt() + 1e-8)
            y = self(z, pts, precision=precision)
        del ones
        return z, loss

    def fit_latents_batch(self, xyz, sdf_target, steps: int = 300, lr: float = 5e-3, clamp: float = 0.1, reg: float = 1e-4,
                          init=None, precision: str = "bf16"):
        """``fit_latent`` for a batch of shapes at once (reconstructing a test set): xyz [B,M,3], sdf_target [B,M] ->
        (latents [B,256], last losses [B]).  Per Adam step: one forward + backward launch per shape, back to back on the
        stream, and one set of [B,256] torch ops; nothing is synchronised until the end.  Tensor-pipe precisions only."""
        prec = PRECISIONS[precision]
        if prec == PRECISIONS["fp32"]:
            raise ValueError("fit_latents_batch runs on the tensor pipe: precision 'bf16' or 'fp16'")
        pts = _as_dev_f32(xyz, self.device)
        if pts.ndim != 3 or pts.shape[2] != 3:
            raise ValueError("expected xyz [B,M,3]")
        B, M = pts.shape[0], pts.shape[1]
        tgt = torch.clamp(_as_dev_f32(sdf_target, self.device, (B, M)), -clamp, clamp)
        z = (torch.zeros((B, LATENT), device=self.device) if init is None
             else _as_dev_f32(init, self.device, (B, LATENT)).clone())
        m, v = torch.zeros_like(z), torch.zeros_like(z)
        loss = torch.zeros(B, device=self.device)
        st = _stream_ptr(self.device.index)
        for it in range(1, steps + 1):
            g = torch.empty_like(z)
            loss = torch.empty(B, dtype=torch.float32, device=self.device)
            check(self._lib.sdfb_decoder_fit_loss_grad_batch(self._h, z.data_ptr(), pts.data_ptr() if M else None, B, M,
                                                             tgt.data_ptr() if M else None, float(clamp), g.data_ptr(),
                                                             loss.data_ptr(), prec, st))
            # loss += reg |z|^2, g += 2 reg z, Adam: one launch (sdfb_latent_adam_step) instead of a dozen elementwise ones
            check(self._lib.sdfb_latent_adam_step(z.data_ptr(), m.data_ptr(), v.data_ptr(), g.data_ptr(), loss.data_ptr(), B, float(lr),
                                                  float(reg), 0.9, 0.999, 1e-8, it, st))
        return z, loss

    def fit_latents_batch_checked(self, *a, **kw):
        """``fit_latents_batch`` followed by ``check()`` (one synchronisation at the end)."""
        out = self.fit_latents_batch(*a, **kw)
        self.check()
        return out

    def extract_surface(self, latent, res: int, precision: str | None = None, indexed: bool = False):
        """decode_grid + marching cubes: triangles [n,3,3] of the zero level set on the res^3 grid
        (the decoder's own sign bit-planes classify the cells); ``indexed=True``: (vertices, faces)."""
        sdf, signs, _ = self.decode_grid_bits(latent, res, mask=False, precision=precision)
        out = extract_surface(sdf, res, 0, sign_words=signs, indexed=indexed)
        self.check()            # the triangle count already synchronised the stream: this only reads the status word
        return out

    def decode_sparse_field(self, latent, res: int, lipschitz: float | None = None, safety: tuple = (2.0, 1.25),
                            precision: str | None = None, local_floor: float = 0.0):
        """(sdf [res,res,res] float32, sign_words int32, stats): the two-level sparse decode of ``sdfb_decode_sparse_field`` -
        ``sdf`` is valid at every node of every cell the surface crosses (uninitialised elsewhere), ``sign_words`` are the
        complete sign bit-planes of the grid; together they are what ``extract_surface(sdf, sign_words=...)`` needs."""
        prec = _prec(precision or self.precision)
        lat = _as_dev_f32(latent, self.device, (LATENT,))
        sdf = torch.empty((res, res, res), dtype=torch.float32, device=self.device)
        signs = torch.empty(((res ** 3 + 31) // 32 + 1,), dtype=torch.int32, device=self.device)
        stats = (C.c_int64 * 8)()
        check(self._lib.sdfb_decode_sparse_field(self._h, lat.data_ptr(), res, C.c_float(0.0 if lipschitz is None else float(lipschitz)),
                                                 C.c_float(float(safety[0])), C.c_float(float(safety[1])), C.c_float(float(local_floor)),
                                                 sdf.data_ptr(), signs.data_ptr(),
                                                 prec, stats, _stream_ptr(self.device.index)))
        keys = ("corner_queries", "blocks_kept", "lattice_queries", "sub_blocks_kept", "fill_queries", "queries")
        st = {k: int(stats[i]) for i, k in enumerate(keys)}
        st.update(dense_queries=res ** 3, lipschitz_level1=stats[6] * 1e-6, lipschitz_level2=stats[7] * 1e-6)
        return sdf, signs, st

    def extract_surface_sparse(self, latent, res: int, lipschitz: float | None = None, precision: str | None = None,
                               return_stats: bool = False, indexed: bool = False, local_floor: float = 0.0):
        """The zero level set on the res^3 grid WITHOUT decoding the whole grid: two-level refinement
        (``decode_sparse_field``), every node decoded at most once, then the DENSE marching-cubes kernels over the complete
        sign bit-planes - with a valid Lipschitz bound the triangle soup equals ``extract_surface``'s bit for bit, order
        included.  ``local_floor`` in (0, 1] lets level 2 use every 8^3 block's own slope estimate (never less than that
        fraction of the global one): a thinner band, fewer queries, less margin."""
        sdf, signs, st = self.decode_sparse_field(latent, res, lipschitz=lipschitz, precision=precision, local_floor=local_floor)
        out = extract_surface(sdf, res, 0, sign_words=signs, indexed=indexed)
        self.check()
        return (out, st) if return_stats else out

    def decode_grid_batch(self, latents, res: int, precision: str | None = None, out: torch.Tensor | None = None) -> torch.Tensor:
        """sdf [B, res, res, res] for latents [B,256] (independent shapes, one C call)."""
        prec = _prec(precision or self.precision)
        lat = _as_dev_f32(latents, self.device)
        if lat.ndim != 2 or lat.shape[1] != LATENT:
            raise ValueError("latents must be [B,256]")
        B = lat.shape[0]
        if out is None:
            out = torch.empty((B, res, res, res), dtype=torch.float32, device=self.device)
        elif out.dtype != torch.float32 or out.device != self.device or not out.is_contiguous() or out.numel() != B * res ** 3:
            raise ValueError("out must be a contiguous float32 CUDA tensor of B * res^3 elements")
        check(self._lib.sdfb_decode_grid_batch(self._h, lat.data_ptr() if B else None, B, res, out.data_ptr() if B else None, prec,
                                               _stream_ptr(self.device.index)))
        return out.view(B, res, res, res)

    def decode_grid_host(self, latent: np.ndarray, res: int, z0: int = 0, z1: int | None = None,
                         mask: bool = False, precision: str | None = None, out: np.ndarray | None = None):
        """Same result as ``decode_grid`` but through the host-buffer entry point: numpy in,
        numpy out, host<->device copies inside the call (the plugin-style call bench.py times)."""
        prec = _prec(precision or self.precision)
        z1 = res if z1 is None else z1
        lat = np.ascontiguousarray(np.asarray(latent, dtype=np.float32).reshape(LATENT))
        if out is None:
            sdf = np.empty((z1 - z0, res, res), dtype=np.float32)
        else:   # caller-owned (ideally pinned) host buffer
            if out.dtype != np.float32 or not out.flags.c_contiguous or out.size != (z1 - z0) * res * res:
                raise ValueError("out must be a C-contiguous float32 array of the slab's size")
            sdf = out.reshape(z1 - z0, res, res)
        halo = mask and z1 < res and z1 > z0
        layers = (z1 if halo else min(z1, res - 1)) - z0
        m = np.empty((max(layers, 0), res - 1, res - 1), dtype=np.uint8) if mask else None
        check(self._lib.sdfb_decode_grid_host(self._h, lat.ctypes.data, res, z0, z1, sdf.ctypes.data,
                                              m.ctypes.data if (m is not None and m.size) else None, prec))
        return (sdf, m) if mask else sdf

    def decode_points_host(self, latent: np.ndarray, xyz: np.ndarray, precision: str | None = None,
                           out: np.ndarray | None = None) -> np.ndarray:
        """Decoder(latent, xyz) with numpy arrays: chunks are copied in, decoded and copied out on three streams.
        ``out`` (optional): a caller-owned, ideally pinned, float32 array of M elements."""
        prec = _prec(precision or self.precision)
        lat = np.ascontiguousarray(np.asarray(latent, dtype=np.float32).reshape(LATENT))
        pts = np.ascontiguousarray(np.asarray(xyz, dtype=np.float32).reshape(-1, 3))
        if out is None:
            out = np.empty(pts.shape[0], dtype=np.float32)
        elif out.dtype != np.float32 or not out.flags.c_contiguous or out.size != pts.shape[0]:
            raise ValueError("out must be a C-contiguous float32 array with one element per point")
        check(self._lib.sdfb_decode_points_host(self._h, lat.ctypes.data, pts.ctypes.data, pts.shape[0],
                                                out.ctypes.data, prec))
        return out

    # ---- status ----------------------------------------------------------------------------
    def check(self) -> None:
        """Waits for the current stream and raises SdfbError if the in-kernel watchdog of any launch made through this
        object tripped (its outputs are then invalid).  The device-path calls are asynchronous: they cannot report their
        own launch, only an earlier one - every call first looks at a host-visible status word the kernels write."""
        check(self._lib.sdfb_decoder_check(self._h, _stream_ptr(self.device.index)))

    def set_watchdog_timeout_ns(self, ns: int) -> None:
        check(self._lib.sdfb_decoder_set_timeout_ns(self._h, int(ns)))

    # ---- diagnostics -----------------------------------------------------------------------
    def debug_pass(self, latent, res: int, pass_index: int, precision: str | None = None) -> torch.Tensor:
        """[128,256] pre-activations (accumulator + bias) of tensor-core pass ``pass_index`` for the
        first 128 grid queries."""
        prec = _prec(precision or self.precision)
        lat = _as_dev_f32(latent, self.device, (LATENT,))
        dump = torch.zeros((128, 256), dtype=torch.float32, device=self.device)
        check(self._lib.sdfb_decode_debug_pass(self._h, lat.data_ptr(), res, pass_index, dump.data_ptr(), prec,
                                               _stream_ptr(self.device.index)))
        return dump

    def last_kernel_ms(self) -> float:
        ms = C.c_float()
        check(self._lib.sdfb_decoder_last_kernel_ms(self._h, C.byref(ms)))
        return float(ms.value)


class LatentDDPM:
    """Latent-space DDPM sampler: MLP denoiser 512 -> 1024x4 -> 256 (epsilon prediction,
    linear beta schedule, 1000 steps, x0-clipped posterior-mean update).

    ``precision``: "fp32" runs the FFMA kernels (carries the 1e-4 criterion); "bf16" / "fp16" run
    all steps of a call in one persistent tcgen05 kernel."""

    def __init__(self, params, device="cuda:0", precision: str = "fp32"):
        self._lib = _lib.load()
        self.device = torch.device("cuda", _device_index(device))
        self.precision = precision
        _prec(precision)
        flat = _flat_params(params, _lib.DDPM_PARAM_FLOATS)
        handle = C.c_void_p()
        check(self._lib.sdfb_ddpm_create(flat.ctypes.data, flat.size, self.device.index, C.byref(handle)))
        self._h = handle

    def close(self):
        if getattr(self, "_h", None):
            self._lib.sdfb_ddpm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def denoise(self, x, t: int, precision: str | None = None) -> torch.Tensor:
        prec = _prec(precision or self.precision)
        xt = _as_dev_f32(x, self.device)
        if xt.ndim != 2 or xt.shape[1] != LATENT:
            raise ValueError("x must be [n,256]")
        eps = torch.empty_like(xt)
        check(self._lib.sdfb_ddpm_denoise(self._h, xt.data_ptr(), int(t), xt.shape[0], eps.data_ptr(), prec,
                                          _stream_ptr(self.device.index)))
        if prec != _lib.PREC_FP32:
            self.last_kernel_ms()       # raises if the fused kernel's watchdog tripped
        return eps

    def sample_latents(self, n: int, x_T=None, noise=None, steps: int = DDPM_STEPS, seed: int = 0,
                       precision: str | None = None, first_latent: int = 0) -> torch.Tensor:
        """x_0 [n,256].  ``noise`` [steps,n,256] (with ``x_T`` [n,256]) is the explicit noise stream of
        the parity tests.  Without ``noise`` the stream is generated in the kernel from ``seed``
        (Philox4x32-10, reproducible on the CPU with oracle/philox.py); ``x_T`` is then optional too.
        ``first_latent`` is the global index of this call's latent 0 in the generator's counters, so shares of
        one batch sampled by different ranks draw the numbers a single call over the whole batch would.
        ``steps`` < 1000 runs only the last ``steps`` steps of the 1000-step chain (truncated, not respaced): a knob
        for parity tests and profiling, not a quality/speed trade - samples need the full 1000."""
        prec = _prec(precision or self.precision)
        if n <= 0:
            raise ValueError("n must be positive")
        if noise is None:
            if x_T is None:
                x = torch.empty((n, LATENT), dtype=torch.float32, device=self.device)
            else:
                x = _as_dev_f32(x_T, self.device, (n, LATENT)).clone()
            check(self._lib.sdfb_ddpm_sample_philox(self._h, x.data_ptr(), int(seed), int(first_latent), n, steps, 1 if x_T is None else 0, prec,
                                                    _stream_ptr(self.device.index)))
            if prec != _lib.PREC_FP32:
                self.last_kernel_ms()
            return x
        if x_T is None:
            raise ValueError("an explicit noise stream needs an explicit x_T")
        x = _as_dev_f32(x_T, self.device, (n, LATENT)).clone()
        nz = _as_dev_f32(noise, self.device, (steps, n, LATENT))
        check(self._lib.sdfb_ddpm_sample(self._h, x.data_ptr(), nz.data_ptr(), n, steps, prec,
                                         _stream_ptr(self.device.index)))
        if prec != _lib.PREC_FP32:
            self.last_kernel_ms()       # waits for the persistent kernel and raises if its watchdog tripped
        return x

    def sample_latents_ddim(self, n: int, steps: int = 50, eta: float = 0.0, x_T=None, noise=None, seed: int = 0,
                            precision: str | None = None, first_latent: int = 0) -> torch.Tensor:
        """x_0 [n,256] by DDIM (Song et al. 2021) on ``steps`` respaced timesteps tau_i = floor(i 1000 / steps) of the
        1000-step chain.  ``eta`` = 0 is deterministic given x_T; ``eta`` = 1 at ``steps`` = 1000 is the DDPM chain of
        ``sample_latents``.  ``noise`` [steps,n,256] (with ``x_T``) is an explicit stream, noise[i] consumed at the step
        from tau_i; it is not needed at ``eta`` = 0.  Without it the stream is generated in the kernel from ``seed``
        (Philox step field tau_i; x_T, when not given, from row 1000, so the same seed starts every step count from the
        same x_T).  ``first_latent`` as in ``sample_latents``.  The rows run are those of ``ddim_schedule``."""
        prec = _prec(precision or self.precision)
        if n <= 0:
            raise ValueError("n must be positive")
        if noise is None and x_T is None:
            x = torch.empty((n, LATENT), dtype=torch.float32, device=self.device)
        elif x_T is None:
            raise ValueError("an explicit noise stream needs an explicit x_T")
        else:
            x = _as_dev_f32(x_T, self.device, (n, LATENT)).clone()
        st = _stream_ptr(self.device.index)
        if noise is None:
            check(self._lib.sdfb_ddpm_sample_ddim_philox(self._h, x.data_ptr(), int(seed), int(first_latent), n, int(steps),
                                                         float(eta), 1 if x_T is None else 0, prec, st))
        else:
            nz = _as_dev_f32(noise, self.device, (int(steps), n, LATENT))
            check(self._lib.sdfb_ddpm_sample_ddim(self._h, x.data_ptr(), nz.data_ptr(), n, int(steps), float(eta), prec, st))
        if prec != _lib.PREC_FP32:
            self.last_kernel_ms()       # waits for the persistent kernel and raises if its watchdog tripped
        return x

    def invert_latents_ddim(self, x0, steps: int = 50, precision: str | None = None) -> torch.Tensor:
        """Deterministic DDIM inversion: the x_T [n,256] (at timestep tau_{steps-1}) from which ``sample_latents_ddim`` with
        the same ``steps`` and ``eta`` = 0 returns to ``x0`` [n,256] (up to the denoiser's sensitivity to its input and
        rounding).  ``x0`` lives in the DDPM's space: a decoder latent (e.g. from ``Decoder.fit_latent``) must be divided by
        ``DDPM_LATENT_SCALE`` first.  x0 is not clipped to [-1, 1] on the way."""
        prec = _prec(precision or self.precision)
        x = _as_dev_f32(x0, self.device).clone()
        if x.ndim != 2 or x.shape[1] != LATENT or x.shape[0] == 0:
            raise ValueError("x0 must be [n,256] with n > 0")
        check(self._lib.sdfb_ddpm_invert_ddim(self._h, x.data_ptr(), x.shape[0], int(steps), prec, _stream_ptr(self.device.index)))
        if prec != _lib.PREC_FP32:
            self.last_kernel_ms()
        return x

    def check(self) -> None:
        """Waits for the current stream; raises SdfbError if the fused sampler's watchdog tripped."""
        check(self._lib.sdfb_ddpm_check(self._h, _stream_ptr(self.device.index)))

    def set_watchdog_timeout_ns(self, ns: int) -> None:
        check(self._lib.sdfb_ddpm_set_timeout_ns(self._h, int(ns)))

    def last_kernel_ms(self) -> float:
        """Device time of the last fused (bf16/fp16) sampler launch; raises SdfbError on a tripped watchdog."""
        ms = C.c_float()
        check(self._lib.sdfb_ddpm_last_kernel_ms(self._h, C.byref(ms)))
        return float(ms.value)

    def sample_latents_seeded_host(self, n: int, seed: int, steps: int = DDPM_STEPS, x_T: np.ndarray | None = None,
                                   precision: str | None = None, first_latent: int = 0) -> np.ndarray:
        """Host-buffer form of the seeded sampler: only x_T (optional) goes in and x_0 comes out."""
        prec = _prec(precision or self.precision)
        x = np.empty((n, LATENT), np.float32) if x_T is None else np.ascontiguousarray(np.asarray(x_T, dtype=np.float32)).copy()
        if x.shape != (n, LATENT):
            raise ValueError("x_T must be [n,256]")
        check(self._lib.sdfb_ddpm_sample_philox_host(self._h, x.ctypes.data, int(seed), int(first_latent), n, steps,
                                                     1 if x_T is None else 0, prec))
        return x

    def sample_latents_host(self, x_T: np.ndarray, noise: np.ndarray, steps: int = DDPM_STEPS,
                            precision: str | None = None) -> np.ndarray:
        prec = _prec(precision or self.precision)
        x = np.ascontiguousarray(np.asarray(x_T, dtype=np.float32)).copy()
        nz = np.ascontiguousarray(np.asarray(noise, dtype=np.float32))
        n = x.shape[0]
        if x.shape != (n, LATENT) or nz.shape != (steps, n, LATENT):
            raise ValueError("expected x_T [n,256] and noise [steps,n,256]")
        check(self._lib.sdfb_ddpm_sample_host(self._h, x.ctypes.data, nz.ctypes.data, n, steps, prec))
        return x


class DDPMTrainer:
    """Training of the latent DDPM's denoiser (SURVEY.md section 8f row N4): one ``step`` = noising, forward, loss, backward
    through all five layers and Adam, on the tensor pipe (``sdfb_ddpm_trainer_step``).  The trainer owns its copy of the
    parameters; ``params()`` downloads them, ``sampler()`` builds a ``LatentDDPM`` from them."""

    def __init__(self, params, device="cuda:0", precision: str = "bf16"):
        self._lib = _lib.load()
        self.device = torch.device("cuda", _device_index(device))
        self.precision = precision
        if precision not in ("bf16", "fp16"):
            raise ValueError("the training step runs on the tensor pipe: precision 'bf16' or 'fp16'")
        flat = _flat_params(params, _lib.DDPM_PARAM_FLOATS)
        handle = C.c_void_p()
        check(self._lib.sdfb_ddpm_trainer_create(flat.ctypes.data, flat.size, self.device.index, _prec(precision), C.byref(handle)))
        self._h = handle

    def close(self):
        if getattr(self, "_h", None):
            self._lib.sdfb_ddpm_trainer_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def step(self, x0, t, eps, lr: float = 1e-4, betas=(0.9, 0.999), adam_eps: float = 1e-8, apply: bool = True,
             return_grads: bool = False):
        """x0 [n,256] clean latents, t [n] int32 in [0, 1000), eps [n,256] noise -> loss [1] (device tensor; nothing is
        synchronised) and, with ``return_grads``, the gradient in the parameter blob's layout.  ``apply=False`` only evaluates."""
        x = _as_dev_f32(x0, self.device)
        e = _as_dev_f32(eps, self.device)
        tt = torch.as_tensor(np.asarray(t) if not isinstance(t, torch.Tensor) else t).to(device=self.device, dtype=torch.int32).contiguous()
        n = x.shape[0]
        if x.shape != (n, LATENT) or e.shape != (n, LATENT) or tt.shape != (n,):
            raise ValueError("expected x0 [n,256], t [n], eps [n,256]")
        loss = torch.empty(1, dtype=torch.float32, device=self.device)
        grads = torch.empty(_lib.DDPM_PARAM_FLOATS, dtype=torch.float32, device=self.device) if return_grads else None
        check(self._lib.sdfb_ddpm_trainer_step(self._h, x.data_ptr(), tt.data_ptr(), e.data_ptr(), n, float(lr), float(betas[0]),
                                               float(betas[1]), float(adam_eps), 1 if apply else 0, loss.data_ptr(),
                                               grads.data_ptr() if grads is not None else None, _stream_ptr(self.device.index)))
        return (loss, grads) if return_grads else loss

    def params(self) -> np.ndarray:
        out = np.empty(_lib.DDPM_PARAM_FLOATS, np.float32)
        check(self._lib.sdfb_ddpm_trainer_get_params(self._h, out.ctypes.data))
        return out

    def sampler(self, precision: str | None = None) -> "LatentDDPM":
        return LatentDDPM(self.params(), device=self.device, precision=precision or self.precision)


class DecoderTrainer:
    """Auto-decoder training (SURVEY.md section 8f row N4): one ``step`` = forward over a batch of shapes' SDF samples,
    clamped-L1 loss, gradients of every decoder weight and bias (weight gradients as tensor-core products contracting over
    the sample index) and Adam (``sdfb_decoder_trainer_step``).  The latents' gradient comes from
    ``Decoder.fit_loss_grad`` / ``fit_latents_batch``.  ``params()`` downloads the weights, ``decoder()`` builds a
    ``Decoder`` from them."""

    def __init__(self, params, device="cuda:0", precision: str = "bf16"):
        self._lib = _lib.load()
        self.device = torch.device("cuda", _device_index(device))
        self.precision = precision
        if precision not in ("bf16", "fp16"):
            raise ValueError("the training step runs on the tensor pipe: precision 'bf16' or 'fp16'")
        flat = _flat_params(params, _lib.DECODER_PARAM_FLOATS)
        handle = C.c_void_p()
        check(self._lib.sdfb_decoder_trainer_create(flat.ctypes.data, flat.size, self.device.index, _prec(precision), C.byref(handle)))
        self._h = handle

    def close(self):
        if getattr(self, "_h", None):
            self._lib.sdfb_decoder_trainer_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def step(self, latents, xyz, sdf_target, clamp: float = 0.1, lr: float = 1e-4, betas=(0.9, 0.999), adam_eps: float = 1e-8,
             apply: bool = True, return_grads: bool = False, return_sdf: bool = False):
        """latents [B,256], xyz [B,P,3], sdf_target [B,P] -> loss [1] (device tensor, nothing synchronised), optionally the
        gradient (decoder blob layout) and the forward values [B,P]."""
        lat = _as_dev_f32(latents, self.device)
        pts = _as_dev_f32(xyz, self.device)
        tgt = _as_dev_f32(sdf_target, self.device)
        if lat.ndim != 2 or lat.shape[1] != LATENT or pts.ndim != 3 or pts.shape[0] != lat.shape[0] or pts.shape[2] != 3 or tgt.shape != pts.shape[:2]:
            raise ValueError("expected latents [B,256], xyz [B,P,3], sdf_target [B,P]")
        B, P = pts.shape[0], pts.shape[1]
        loss = torch.empty(1, dtype=torch.float32, device=self.device)
        grads = torch.empty(_lib.DECODER_PARAM_FLOATS, dtype=torch.float32, device=self.device) if return_grads else None
        sdf = torch.empty((B, P), dtype=torch.float32, device=self.device) if return_sdf else None
        check(self._lib.sdfb_decoder_trainer_step(self._h, lat.data_ptr(), pts.data_ptr(), tgt.data_ptr(), B, P, float(clamp), float(lr),
                                                  float(betas[0]), float(betas[1]), float(adam_eps), 1 if apply else 0, loss.data_ptr(),
                                                  grads.data_ptr() if grads is not None else None,
                                                  sdf.data_ptr() if sdf is not None else None, _stream_ptr(self.device.index)))
        out = (loss,)
        if return_grads:
            out += (grads,)
        if return_sdf:
            out += (sdf,)
        return out if len(out) > 1 else loss

    def params(self) -> np.ndarray:
        out = np.empty(_lib.DECODER_PARAM_FLOATS, np.float32)
        check(self._lib.sdfb_decoder_trainer_get_params(self._h, out.ctypes.data))
        return out

    def decoder(self, precision: str | None = None) -> "Decoder":
        return Decoder(self.params(), device=self.device, precision=precision or self.precision)


class _DevArray:
    """A device pointer owned by the C library, seen by torch without a copy (``__cuda_array_interface__``)."""

    def __init__(self, ptr: int, shape, typestr: str):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}


class Comm:
    """Ranks of one node, one process per GPU (SURVEY.md section 8e): wraps ``sdfb_comm`` - NCCL for the barrier and the
    in-place slab all-gather, and a symmetric device buffer mapped into every rank through CUDA IPC into which finished
    sub-slabs are pushed by the copy engines while the decoder kernel keeps all SMs.  Bootstrapped over an initialised
    ``torch.distributed`` group (only to hand rank 0's NCCL id to the others)."""

    def __init__(self, device="cuda:0", group=None):
        import torch.distributed as dist
        self._lib = _lib.load()
        self.device = torch.device("cuda", _device_index(device))
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        ident = np.zeros(128, np.uint8)
        if self.rank == 0 and self.world > 1:
            check(self._lib.sdfb_comm_unique_id(ident.ctypes.data))
        if self.world > 1:
            t = torch.from_numpy(ident)
            if dist.get_backend(group) == "nccl":
                t = t.to(self.device)
            src = dist.get_global_rank(group, 0) if group is not None else 0
            dist.broadcast(t, src=src, group=group)
            ident = t.cpu().numpy().copy()
        handle = C.c_void_p()
        with torch.cuda.device(self.device):
            check(self._lib.sdfb_comm_create(ident.ctypes.data, self.world, self.rank, self.device.index, C.byref(handle)))
        self._h = handle

    def close(self):
        if getattr(self, "_h", None):
            self._lib.sdfb_comm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def barrier(self) -> None:
        check(self._lib.sdfb_comm_barrier(self._h, _stream_ptr(self.device.index)))

    def allgather_slabs(self, full: torch.Tensor) -> torch.Tensor:
        """In-place NCCL all-gather: ``full`` is split into ``world`` equal leading blocks, rank r's is already filled."""
        if not full.is_contiguous() or full.device != self.device or full.shape[0] % self.world:
            raise ValueError("full must be a contiguous CUDA tensor whose leading size is a multiple of the world size")
        per = full.numel() * full.element_size() // self.world
        check(self._lib.sdfb_allgather_slabs(self._h, full.data_ptr(), per, _stream_ptr(self.device.index)))
        return full

    def decode_grid_sharded(self, decoder: "Decoder", latent, res: int, mask: bool = False, precision: str | None = None,
                            sub_planes: int = 0):
        """BASELINE configs[4]: (sdf [res,res,res], mask_words int32 [world, words_per_rank] or None).  Both are views of
        the communicator's symmetric buffer: valid until the next sharded decode on it.  See ``sdfb_decode_grid_sharded``
        (include/sdfb200.h) for the block layout of the packed mask and ``unpack_mask_blocks`` for the uint8 form."""
        prec = _prec(precision or decoder.precision)
        lat = _as_dev_f32(latent, self.device, (LATENT,))
        sdf_p, mask_p, words = C.c_void_p(), C.c_void_p(), C.c_size_t()
        check(self._lib.sdfb_decode_grid_sharded(decoder._h, self._h, lat.data_ptr(), res, 1 if mask else 0, int(sub_planes), prec,
                                                 C.byref(sdf_p), C.byref(mask_p), C.byref(words), _stream_ptr(self.device.index)))
        sdf = torch.as_tensor(_DevArray(sdf_p.value, (res, res, res), "<f4"), device=self.device)
        mw = None
        if mask:
            mw = torch.as_tensor(_DevArray(mask_p.value, (self.world, words.value), "<i4"), device=self.device)
        return sdf, mw


def unpack_mask_blocks(mask_words: torch.Tensor, res: int) -> torch.Tensor:
    """[world, words_per_rank] packed mask blocks of ``Comm.decode_grid_sharded`` -> uint8 [(res-1)^3] cell mask."""
    world = mask_words.shape[0]
    per = -(-res // world)
    cells = (res - 1) * (res - 1)
    shifts = torch.arange(32, device=mask_words.device, dtype=torch.int32)
    out = []
    for r in range(world):
        z0 = min(r * per, res)
        layers = max(min(z0 + per, res - 1) - z0, 0)
        if layers == 0:
            continue
        nw = (layers * cells + 31) // 32
        bits = ((mask_words[r, :nw].unsqueeze(1) >> shifts) & 1).to(torch.uint8).reshape(-1)[: layers * cells]
        out.append(bits.view(layers, res - 1, res - 1))
    return torch.cat(out) if out else torch.empty((0, res - 1, res - 1), dtype=torch.uint8, device=mask_words.device)


# ---- functional spellings named in the north star ---------------------------------------------
def decode_grid(decoder: Decoder, z, res: int, **kw):
    return decoder.decode_grid(z, res, **kw)


def sample_latents(ddpm: LatentDDPM, n: int, **kw):
    return ddpm.sample_latents(n, **kw)


def ddim_schedule(steps: int, eta: float, inverse: bool = False):
    """The rows a respaced call runs, in execution order (``sdfb_ddim_schedule``; no device needed):
    timesteps int32 [steps] and coefficients float32 [steps, 8] = (sra, srm1, c1, c2, c3, sigma, clamp, 0)."""
    lib = _lib.load()
    ts = np.zeros(int(steps) if int(steps) > 0 else 0, np.int32)
    coef = np.zeros((ts.size, 8), np.float32)
    check(lib.sdfb_ddim_schedule(int(steps), float(eta), 1 if inverse else 0, ts.ctypes.data, coef.ctypes.data))
    return ts, coef


def philox_normal(seed: int, n: int, t0: int, t1: int, device="cuda:0", first_latent: int = 0) -> torch.Tensor:
    """The sampler's noise stream: normals of steps [t0, t1) for latents [first_latent, first_latent + n),
    [(t1-t0), n, 256]."""
    lib = _lib.load()
    dev = torch.device("cuda", _device_index(device))
    out = torch.empty((t1 - t0, n, LATENT), dtype=torch.float32, device=dev)
    if out.numel():
        with torch.cuda.device(dev):
            check(lib.sdfb_philox_normal(int(seed), int(first_latent), n, t0, t1, out.data_ptr(), _stream_ptr(dev.index)))
    return out


def weld(tris: torch.Tensor, keys: torch.Tensor, res: int):
    """Triangle soup [n,3,3] + grid-edge keys [n,3] of a res^3 grid -> indexed mesh (vertices [V,3] in ascending key order,
    faces [n,3] int64).  ``sdfb_mc_weld_count`` / ``_fill``: a bitmap over the grid's edges, ranked by a scan."""
    lib = _lib.load()
    n = int(tris.shape[0])
    t, k = tris.contiguous(), keys.contiguous()
    with torch.cuda.device(tris.device):
        nbytes = C.c_size_t()
        check(lib.sdfb_mc_weld_workspace_bytes(int(res), C.byref(nbytes)))
        ws = torch.empty((nbytes.value,), dtype=torch.uint8, device=tris.device)
        nv = C.c_int64()
        st = _stream_ptr(tris.device.index)
        check(lib.sdfb_mc_weld_count(k.data_ptr() if n else None, n, int(res), ws.data_ptr(), nbytes.value, C.byref(nv), st))
        verts = torch.empty((nv.value, 3), dtype=torch.float32, device=tris.device)
        faces = torch.empty((n, 3), dtype=torch.int64, device=tris.device)
        if n:
            check(lib.sdfb_mc_weld_fill(t.data_ptr(), k.data_ptr(), n, int(res), ws.data_ptr(), verts.data_ptr(), faces.data_ptr(), st))
    return verts, faces


def extract_surface(sdf: torch.Tensor, res: int | None = None, z0: int = 0, sign_words: torch.Tensor | None = None,
                    indexed: bool = False):
    """Marching cubes on a [nz,ny,nx] float32 CUDA field -> triangles [n,3,3] (x,y,z), cell order, normals
    from inside (sdf < 0) to outside.  ``res``/``z0`` place a slab in the res^3 grid of rule A1 (default:
    the field is the whole grid); ``sign_words`` are the bit-planes from ``Decoder.decode_grid_bits``.
    ``indexed=True`` returns (vertices [V,3], faces [n,3]) instead: vertices on the same grid edge are merged."""
    lib = _lib.load()
    if sdf.ndim != 3 or sdf.dtype != torch.float32 or not sdf.is_cuda:
        raise ValueError("sdf must be a 3-D float32 CUDA tensor")
    s = sdf.contiguous()
    nz, ny, nx = s.shape
    res = nx if res is None else res
    if min(nz, ny, nx) < 2:
        empty = torch.empty((0, 3, 3), dtype=torch.float32, device=s.device)
        return (empty.reshape(0, 3), torch.empty((0, 3), dtype=torch.int64, device=s.device)) if indexed else empty
    with torch.cuda.device(s.device):
        nbytes = C.c_size_t()
        check(lib.sdfb_mc_workspace_bytes(nz, ny, nx, C.byref(nbytes)))
        ws = torch.empty((nbytes.value,), dtype=torch.uint8, device=s.device)
        n = C.c_int64()
        st = _stream_ptr(s.device.index)
        check(lib.sdfb_mc_count(s.data_ptr(), sign_words.data_ptr() if sign_words is not None else None, nz, ny, nx,
                                ws.data_ptr(), nbytes.value, C.byref(n), st))
        tris = torch.empty((n.value, 3, 3), dtype=torch.float32, device=s.device)
        keys = torch.empty((n.value, 3), dtype=torch.int64, device=s.device) if indexed else None
        if n.value:
            check(lib.sdfb_mc_generate(s.data_ptr(), nz, ny, nx, res, z0, ws.data_ptr(), tris.data_ptr(),
                                       keys.data_ptr() if indexed else None, st))
    return weld(tris, keys, res) if indexed else tris


def grid_points(res: int, z0: int = 0, z1: int | None = None, device="cuda:0") -> torch.Tensor:
    """xyz [(z1-z0)*res*res, 3] of the grid nodes (x fastest), bit-exact rule A1."""
    lib = _lib.load()
    dev = torch.device("cuda", _device_index(device))
    z1 = res if z1 is None else z1
    out = torch.empty(((z1 - z0) * res * res, 3), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        check(lib.sdfb_grid_points(res, z0, z1, out.data_ptr(), _stream_ptr(dev.index)))
    return out


def sign_change_mask(sdf: torch.Tensor) -> torch.Tensor:
    """A4 on a [nz,ny,nx] float32 CUDA tensor -> uint8 [(nz-1),(ny-1),(nx-1)]."""
    lib = _lib.load()
    if sdf.ndim != 3 or sdf.dtype != torch.float32 or not sdf.is_cuda:
        raise ValueError("sdf must be a 3-D float32 CUDA tensor")
    s = sdf.contiguous()
    nz, ny, nx = s.shape
    out = torch.empty((max(nz - 1, 0), max(ny - 1, 0), max(nx - 1, 0)), dtype=torch.uint8, device=s.device)
    if out.numel():
        with torch.cuda.device(s.device):
            check(lib.sdfb_sign_change_mask(s.data_ptr(), nz, ny, nx, out.data_ptr(), _stream_ptr(s.device.index)))
    return out
