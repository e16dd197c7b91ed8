"""Exact tests of the fused decoder (K1) on an integer-valued network (oracle/integer_decoder.py).

On that network every sum the decoder forms is exact in fp32 whatever its order, and every 16-bit rounding is
deterministic, so the pre-activation x = h7 . w8 + b8 has one correct value at every query.  The reference
(``integer_decoder.forward``, float64, checking its own premise) gives it; the kernel's output y = tanhf(x) must
then satisfy, at every node of every field:

  * sign(y) == sign(x) and y == 0 exactly where x == 0;
  * |y - tanh(x)| <= 2 ulp(fp32), the documented maximum error of CUDA's tanhf.  Where |x| <= 4 (at least
    90 % of every field here, asserted) one granule of x (2^-8) moves tanh by far more than that, so the bound
    leaves no room for a wrong x.

Per-pass dumps (pre-activations, no tanh) are compared with torch.equal.  A mismatch names the wrong nodes and
where the persistent schedule put them (128-row half tile, pair tile, CTA pair, rank, round); a wrong node in
the first tile of a grid launch also gets the first wrong tensor-core pass.
"""
import numpy as np
import pytest
import torch

import oracle
from oracle import integer_decoder as I

LATENTS = (0, 1, 2)             # 0 is the zero latent
PRECS = ("bf16", "fp16")
PASS_LAYER = [(1, 0), (1, 256), (2, 0), (2, 256), (3, 0), (4, 0), (4, 256), (5, 0), (5, 256), (6, 0), (6, 256),
              (7, 0), (7, 256)]            # tensor-core pass -> (layer, first column)
POINT_COUNTS = (1, 127, 128, 129, 255, 256, 257, 5000, 3 * 2 ** 20 + 77)


# ---------------------------------------------------------------------------------------------------------------
# helpers
def assert_nondegenerate(x: torch.Tensor, stats: I.Stats, what: str):
    inside = float((x < 0).double().mean())
    small = float((x.abs() <= 4).double().mean())
    assert 0.2 <= inside <= 0.8, f"{what}: {inside:.3f} of the field inside"
    assert small >= 0.9, f"{what}: |x| <= 4 at only {small:.3f} of the nodes"
    for layer in range(8):
        a = stats.active_fraction(layer)
        assert 0.2 <= a <= 0.8, f"{what}: layer {layer} active fraction {a:.3f}"
        assert stats.dead_queries[layer] == 0, f"{what}: layer {layer} has no active unit at some queries"


def schedule(m: torch.Tensor, M: int, num_sms: int) -> str:
    """Where the persistent kernel's schedule puts queries m of a launch of M queries (fused_decoder.cu: pair tiles
    of 256 rows, tile t on pair t % npairs in round t // npairs, rank (m % 256) // 128).  M = None: the call
    split the queries over several launches of its own choosing; only the indices are given."""
    if M is None:
        return "(queries of a call that made its own launches) " + ", ".join(str(q) for q in m.tolist())
    tiles = (M + 255) // 256
    npairs = min(tiles, num_sms // 2)
    out = []
    for q in m.tolist():
        t = q // 256
        out.append(f"query {q}: half-tile {q // 128}, tile {t}, pair {t % npairs}, rank {(q % 256) // 128}, "
                   f"round {t // npairs} of {(tiles - t % npairs + npairs - 1) // npairs}")
    return f"(launch of {M} queries, {npairs} pairs)\n    " + "\n    ".join(out)


def tanh_check(y: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """Boolean [n]: y (fp32, the kernel's tanhf(x)) is right for the exact pre-activation x (float64)."""
    t = torch.tanh(x)
    t32 = t.to(torch.float32).abs()
    ulp = (torch.nextafter(t32, torch.full_like(t32, float("inf"))) - t32).double()
    close = (y.double() - t).abs() <= 2 * ulp
    return close & (torch.sign(y.double()) == torch.sign(x)) & ((y == 0) == (x == 0))


def first_wrong_pass(dec, latent, res: int, prec: str) -> str:
    """Compares the 13 pass dumps of the first 128 grid queries with the reference: the first wrong one."""
    _, pre = I.forward(latent, I.grid_xyz(res, 0, 128, "cuda"), prec, preacts=True)
    for p, (layer, c0) in enumerate(PASS_LAYER):
        want = pre[layer][:, c0:c0 + 256]
        got = dec.debug_pass(latent, res, p, precision=prec)[:, :want.shape[1]].double()
        bad = (got != want).nonzero()
        if bad.numel():
            r, c = bad[0].tolist()
            return (f"first wrong pass {p} (layer {layer}, columns {c0}..{c0 + 255}): {bad.shape[0]} wrong values, "
                    f"first at row {r}, column {c0 + c}: {got[r, c].item()} instead of {want[r, c].item()}")
    return "all 13 passes of the first 128 queries are right"


def check_field(y: torch.Tensor, x: torch.Tensor, M: int, what: str, offset: int = 0, grid=None):
    """The kernel's outputs y [n] against exact pre-activations x [n]; y[i] is query offset + i of a launch of M
    queries.  grid = (dec, latent, res, prec) for a grid launch starting at query 0 (adds the first wrong pass)."""
    y, x = y.reshape(-1), x.reshape(-1)
    assert y.shape == x.shape, (y.shape, x.shape)
    ok = tanh_check(y, x)
    if bool(ok.all()):
        return
    bad = (~ok).nonzero().squeeze(1)
    idx = bad[:6]
    vals = "; ".join(f"[{i}] y {y[i].item()!r} for x {x[i].item()!r}" for i in idx.tolist())
    msg = f"{what}: {bad.numel()} of {y.numel()} nodes wrong, first {idx.tolist()}: {vals}\n  "
    msg += schedule(idx + offset, M, torch.cuda.get_device_properties(y.device).multi_processor_count)
    if grid is not None and offset == 0 and int(bad[0]) < 256:
        msg += "\n  " + first_wrong_pass(*grid)
    raise AssertionError(msg)


def torch_mask(inside: torch.Tensor) -> torch.Tensor:
    """oracle.sign_change_mask from a boolean [nz, ny, nx] inside field, on the device."""
    nz, ny, nx = inside.shape
    any_in = torch.zeros((nz - 1, ny - 1, nx - 1), dtype=torch.bool, device=inside.device)
    all_in = torch.ones_like(any_in)
    for dz in (0, 1):
        for dy in (0, 1):
            for dx in (0, 1):
                c = inside[dz:nz - 1 + dz, dy:ny - 1 + dy, dx:nx - 1 + dx]
                any_in |= c
                all_in &= c
    return (any_in & ~all_in).to(torch.uint8)


def pack_bits(b: torch.Tensor) -> torch.Tensor:
    """bool [n] -> int32 words, bit (i & 31) of word i >> 5 (the decoder's sign and mask words)."""
    b = b.reshape(-1)
    pad = (-b.numel()) % 32
    w = torch.cat([b, b.new_zeros(pad)]).view(-1, 32).to(torch.int64)
    v = (w << torch.arange(32, device=b.device)).sum(1)
    return torch.where(v >= 2 ** 31, v - 2 ** 32, v).to(torch.int32)


def check_words(got: torch.Tensor, want_bits: torch.Tensor, M: int, what: str, offset: int = 0):
    """Packed words against the bits they must hold; a mismatch names the first wrong bits' queries."""
    want = pack_bits(want_bits)
    got = got[:want.numel()]
    if torch.equal(got, want):
        return
    words = (got != want).nonzero().squeeze(1)
    w = int(words[0])
    diff = int(got[w]) ^ int(want[w])
    nodes = torch.tensor([32 * w + k for k in range(32) if (diff >> k) & 1], device=got.device)
    msg = (f"{what}: {words.numel()} of {want.numel()} words wrong; word {w} differs at bits of nodes "
           f"{nodes.tolist()}\n  ")
    raise AssertionError(msg + schedule(nodes[:6] + offset, M, torch.cuda.get_device_properties(got.device).multi_processor_count))


# ---------------------------------------------------------------------------------------------------------------
# CPU: the reference itself
@pytest.mark.parametrize("latent", LATENTS)
def test_reference_equals_frozen_oracle(latent):
    """The exact reference, rounded to fp32, equals the frozen oracle bit for bit - outputs and the pre-activations
    of layers 1..7 - at bf16, fp16 (decoder_forward_lowp) and fp32 (decoder_forward).  So the oracle's own fp32 sums
    are order-free on this network too."""
    P = I.integer_decoder_weights()
    z = I.integer_latent(latent)
    pts = np.concatenate([I.dyadic_points(2500, seed=latent), oracle.grid_points(65, 31, 32)[::8]])
    for prec, lowp in (("bf16", torch.bfloat16), ("fp16", torch.float16)):
        pre_o = []
        want = oracle.decoder_forward_lowp(z, pts, params=P, lowp=lowp, preacts=pre_o)
        x, pre = I.forward(z, pts, prec, preacts=True)
        assert np.array_equal(torch.tanh(x.float()).numpy(), want), prec
        for layer in range(1, 8):
            assert np.array_equal(pre[layer].float().numpy(), pre_o[layer - 1]), (prec, layer)
    x = I.forward(z, pts, "fp32")
    assert np.array_equal(torch.tanh(x.float()).numpy(), oracle.decoder_forward(z, pts, params=P))


def test_network_is_integer_valued():
    P = I.integer_decoder_weights()
    assert len(P) == 9 and oracle.flatten_params(P).size == 1839358
    for li, (w, b) in enumerate(P[:8]):
        assert np.array_equal(w, np.round(w)) and np.array_equal(b, np.round(b)), li
    w0, w4 = P[0][0], P[4][0]
    assert set(np.unique(w0[:, :256])) <= {-1, 0, 1} and np.all(w0[:, 256:] % 256 == 0)
    assert set(np.unique(w4[:, 253:509])) <= {-1, 0, 1} and np.all(w4[:, 509:] % 256 == 0)
    for li in (1, 2, 3, 5, 6, 7):
        assert set(np.unique(P[li][0])) <= {-1, 0, 1}
    w8, b8 = P[8]
    assert np.all(w8 != 0) and np.array_equal(w8 * 256, np.round(w8 * 256)) and float(b8[0] * 256) == round(float(b8[0] * 256))
    for k in (0, 1, 2):
        z = I.integer_latent(k)
        assert np.array_equal(z, np.round(z)) and (k == 0) == (not z.any())
    for res in (65, 129, 257, 513):     # grid coordinates are multiples of 1/256: exact in bf16 and fp16
        c = oracle.axis_coords(res).astype(np.float64)
        assert np.array_equal(c * 256, np.round(c * 256))
        assert np.array_equal(I.grid_xyz(res, 0, res).numpy()[:, 0], c)


@pytest.mark.parametrize("prec,latent", (("bf16", 1), ("fp16", 2), ("fp32", 0)))
def test_premise_and_nondegeneracy_65(prec, latent):
    st = I.Stats()
    x = I.forward_grid(I.integer_latent(latent), 65, prec, stats=st)
    print(f"65^3 {prec} latent {latent}: {st.summary()}")
    assert_nondegenerate(x, st, f"65^3 {prec} latent {latent}")


def test_premise_nondegeneracy_and_zeros_129():
    """The 129^3 field of latent 1 (bf16) has exact zeros - x == 0 at >= 1000 nodes - besides passing the premise
    and non-degeneracy checks."""
    st = I.Stats()
    x = I.forward_grid(I.integer_latent(1), 129, "bf16", stats=st)
    print(f"129^3 bf16 latent 1: {st.summary()}; zeros {int((x == 0).sum())}")
    assert_nondegenerate(x, st, "129^3 bf16 latent 1")
    assert int((x == 0).sum()) >= 1000


# ---------------------------------------------------------------------------------------------------------------
# GPU
_REF = {}


def ref_grid(latent: int, res: int, prec: str) -> torch.Tensor:
    """Exact x of the whole res^3 grid on the device (cached); premise and non-degeneracy asserted."""
    key = (latent, res, prec)
    if key not in _REF:
        st = I.Stats()
        x = I.forward_grid(I.integer_latent(latent), res, prec, device="cuda", chunk=1 << 18, stats=st)
        print(f"{res}^3 {prec} latent {latent}: {st.summary()}")
        assert_nondegenerate(x, st, f"{res}^3 {prec} latent {latent}")
        _REF[key] = x
    return _REF[key]


_PTS = {}


def ref_points(latent: int, prec: str):
    """The dyadic points of the points-mode tests and their exact x (cached)."""
    if "xyz" not in _PTS:
        _PTS["xyz"] = I.dyadic_points(max(POINT_COUNTS), seed=7)
    key = (latent, prec)
    if key not in _PTS:
        _PTS[key] = I.forward_points(I.integer_latent(latent), _PTS["xyz"], prec, device="cuda", chunk=1 << 18)
    return _PTS["xyz"], _PTS[key]


@pytest.fixture(scope="module")
def idec(pkg):
    dec = pkg.Decoder(oracle.flatten_params(I.integer_decoder_weights()), device="cuda:0", precision="bf16")
    yield dec
    dec.close()
    _REF.clear()
    _PTS.clear()


@pytest.mark.gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("res", (65, 129))
def test_pass_dumps_exact(idec, prec, res):
    """All 13 tensor-core passes of the first 128 grid queries equal the reference's pre-activations exactly."""
    for latent in (0, 1):
        z = I.integer_latent(latent)
        _, pre = I.forward(z, I.grid_xyz(res, 0, 128, "cuda"), prec, preacts=True)
        for p, (layer, c0) in enumerate(PASS_LAYER):
            want = pre[layer][:, c0:c0 + 256]
            dump = idec.debug_pass(z, res, p, precision=prec)
            got = dump[:, :want.shape[1]].double()
            if not torch.equal(got, want):
                bad = (got != want).nonzero()
                r, c = bad[0].tolist()
                raise AssertionError(f"latent {latent} {prec} res {res}: pass {p} (layer {layer}, columns {c0}..) has "
                                     f"{bad.shape[0]} wrong values; first at query {r} (tile 0, pair 0, rank 0), "
                                     f"column {c0 + c}: {got[r, c].item()} instead of {want[r, c].item()}")
            if layer == 3:       # L3's padding columns: no weights, no bias
                assert not bool(dump[:, want.shape[1]:].any()), "pass 4 padding columns are not zero"


@pytest.mark.gpu
@pytest.mark.parametrize("prec", PRECS)
def test_points_exact(idec, prec):
    """Points mode at ragged and multi-round sizes, three latents (one of them zero), and the batch-of-shapes call."""
    for latent in LATENTS:
        z = I.integer_latent(latent)
        xyz, x = ref_points(latent, prec)
        for M in POINT_COUNTS:
            y = idec(z, xyz[:M], precision=prec)
            check_field(y, x[:M], M, f"points latent {latent} {prec} M={M}")
    M = 1000
    zz = np.stack([I.integer_latent(k) for k in LATENTS])
    pp = np.stack([I.dyadic_points(M, seed=100 + k) for k in LATENTS])
    yb = idec(zz, pp, precision=prec)
    for k in LATENTS:
        x = I.forward(I.integer_latent(k), torch.from_numpy(pp[k]).double().cuda(), prec)
        check_field(yb[k], x, M, f"batch of shapes, shape {k} {prec}")


@pytest.mark.gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("res", (129, 257, 513))
def test_full_grid_exact(idec, prec, res):
    """The whole res^3 field, its slabs (starting mid sign word, with and without the halo plane), the sign bit-planes
    and the u8 / packed masks, all against the exact reference."""
    latent = 1
    z = I.integer_latent(latent)
    x = ref_grid(latent, res, prec)
    plane = res * res
    sdf = idec.decode_grid(z, res, precision=prec)
    check_field(sdf, x, res ** 3, f"{res}^3 {prec} field", grid=(idec, z, res, prec))
    if res == 513:
        same = torch.equal(sdf.reshape(-1), torch.tanh(x.float()))
        print(f"{res}^3 {prec}: kernel tanhf == torch.tanh(fp32 x) on the device at every node: {same}")
    inside = (x < 0).view(res, res, res)
    # slabs: z0 * res^2 is odd (res^2 is odd), so a slab starts in the middle of a 32-query sign word
    for z0, z1 in ((1, 6), (res // 2 + 1, res // 2 + 4), (res - 5, res)):
        for mask in (False, True):
            halo = 1 if (mask and z1 < res) else 0
            M = (z1 - z0 + halo) * plane
            out = idec.decode_grid(z, res, z0, z1, mask=mask, precision=prec)
            s = out[0] if mask else out
            check_field(s, x[z0 * plane:z1 * plane], M, f"{res}^3 {prec} slab [{z0}, {z1}) mask={mask}")
            if mask:
                want = torch_mask(inside[z0:z1 + halo])
                m = out[1]
                if not torch.equal(m, want):
                    c = (m != want).nonzero()[0].tolist()
                    raise AssertionError(f"{res}^3 {prec} slab [{z0}, {z1}): u8 mask wrong at {(m != want).sum().item()} "
                                         f"cells, first (z, y, x) = {c} of the slab")
        sdf_b, signs, mw = idec.decode_grid_bits(z, res, z0, z1, precision=prec)
        halo = 1 if z1 < res else 0
        M = (z1 - z0 + halo) * plane
        check_field(sdf_b, x[z0 * plane:z1 * plane], M, f"{res}^3 {prec} decode_grid_bits [{z0}, {z1}) values")
        check_words(signs, inside[z0:z1 + halo], M, f"{res}^3 {prec} sign bit-planes [{z0}, {z1})")
        check_words(mw, torch_mask(inside[z0:z1 + halo]).bool(), M, f"{res}^3 {prec} packed mask [{z0}, {z1})")
    # the whole grid's sign planes and both masks
    _, m = idec.decode_grid(z, res, mask=True, precision=prec)
    want_mask = torch_mask(inside)
    assert torch.equal(m, want_mask), f"{res}^3 {prec}: u8 mask wrong at {(m != want_mask).sum().item()} cells"
    _, signs, mw = idec.decode_grid_bits(z, res, precision=prec)
    check_words(signs, inside, res ** 3, f"{res}^3 {prec} sign bit-planes")
    check_words(mw, want_mask.bool(), res ** 3, f"{res}^3 {prec} packed mask")


@pytest.mark.gpu
def test_host_entry_points_exact(idec):
    """decode_grid_host (z-chunks, halo, mask), decode_points_host above 2^21 points, decode_grid_batch."""
    prec = "bf16"
    res, plane = 257, 257 * 257
    z = I.integer_latent(2)
    x = ref_grid(2, res, prec)
    inside = (x < 0).view(res, res, res)
    for z0, z1 in ((0, res), (3, 200)):
        sdf, m = idec.decode_grid_host(z, res, z0, z1, mask=True, precision=prec)
        check_field(torch.from_numpy(sdf).cuda(), x[z0 * plane:z1 * plane], None, f"decode_grid_host [{z0}, {z1})")
        halo = 1 if z1 < res else 0
        assert torch.equal(torch.from_numpy(m).cuda(), torch_mask(inside[z0:z1 + halo])), f"decode_grid_host [{z0}, {z1}) mask"
    xyz, xp = ref_points(1, prec)
    M = 2 ** 21 + 2 ** 20 + 77
    y = idec.decode_points_host(I.integer_latent(1), xyz[:M], precision=prec)
    check_field(torch.from_numpy(y).cuda(), xp[:M], None, "decode_points_host")
    zz = np.stack([I.integer_latent(k) for k in LATENTS])
    out = idec.decode_grid_batch(zz, 129, precision=prec)
    for k in LATENTS:
        check_field(out[k], ref_grid(k, 129, prec), 129 ** 3, f"decode_grid_batch shape {k}",
                    grid=(idec, I.integer_latent(k), 129, prec))


@pytest.mark.gpu
def test_ffma_path_exact(idec):
    """precision="fp32" (the FFMA kernels): points and the 129^3 grid equal the unrounded reference."""
    for latent in (0, 1):
        z = I.integer_latent(latent)
        xyz, x = ref_points(latent, "fp32")
        for M in (129, 5000, 70000):
            check_field(idec(z, xyz[:M], precision="fp32"), x[:M], M, f"fp32 points latent {latent} M={M}")
    check_field(idec.decode_grid(I.integer_latent(1), 129, precision="fp32"), ref_grid(1, 129, "fp32"), 129 ** 3,
                "fp32 129^3 field")


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ("bf16", "fp16", "fp32"))
def test_exact_zeros(pkg, idec, prec):
    """On the 129^3 field with exact zeros: the sign planes count 0 as outside, the mask is oracle.sign_change_mask of
    the field and the surface equals oracle.marching_cubes bit for bit - vertices then land on nodes (t = 0 or 1)."""
    res = 129
    z = I.integer_latent(1)
    x = ref_grid(1, res, prec)
    sdf, signs, _ = idec.decode_grid_bits(z, res, precision=prec)
    check_field(sdf, x, res ** 3, f"{res}^3 {prec} field with zeros", grid=(idec, z, res, prec) if prec != "fp32" else None)
    zeros = int((sdf == 0).sum())
    assert zeros >= 1000, zeros
    check_words(signs, sdf.reshape(-1) < 0, res ** 3, f"{res}^3 {prec} sign planes with zeros")
    f = sdf.cpu().numpy()
    _, m = idec.decode_grid(z, res, mask=True, precision=prec)
    assert np.array_equal(m.cpu().numpy(), oracle.sign_change_mask(f))
    tris = idec.extract_surface(z, res, precision=prec).cpu().numpy()
    want = oracle.marching_cubes(f)
    assert tris.shape == want.shape and np.array_equal(tris.view(np.uint32), want.view(np.uint32))
    c = oracle.axis_coords(res)
    on_node = np.isin(want.reshape(-1, 3), c).all(axis=1)
    print(f"{res}^3 {prec}: {zeros} zero nodes, {want.shape[0]} triangles, {int(on_node.sum())} vertices on nodes")
    assert on_node.sum() > 0
