"""Marching cubes (SURVEY.md section 8f, N1): generated case tables, the numpy oracle, and - on the GPU -
the CUDA extraction compared bit for bit with the oracle."""
import os

import numpy as np
import pytest
import torch

import importlib.util

import oracle
from oracle import mc_tables

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _generator():
    """tools/gen_mc_tables.py, the product's build tool that writes csrc/mc_tables.h and oracle/mc_tables.npz"""
    spec = importlib.util.spec_from_file_location("gen_mc_tables", os.path.join(ROOT, "tools", "gen_mc_tables.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _sphere(res, r=0.6, c=(0.05, -0.1, 0.02)):
    a = oracle.axis_coords(res)
    zz, yy, xx = np.meshgrid(a, a, a, indexing="ij")
    return (np.sqrt((xx - c[0]) ** 2 + (yy - c[1]) ** 2 + (zz - c[2]) ** 2) - r).astype(np.float32)


def test_tables_are_consistent_and_header_is_current():
    assert mc_tables.MC_MAX_TRI == 5
    assert mc_tables.MC_NTRI[0] == 0 and mc_tables.MC_NTRI[255] == 0
    for case in range(256):
        n = mc_tables.MC_NTRI[case]
        used = mc_tables.MC_TRI[case, : 3 * n]
        assert (used >= 0).all() and (mc_tables.MC_TRI[case, 3 * n:] == -1).all()
        inside = [(case >> i) & 1 for i in range(8)]
        crossed = {e for e, (a, b) in enumerate(mc_tables.EDGES) if inside[a] != inside[b]}
        assert set(int(e) for e in used) == crossed          # every crossed edge carries a vertex, no other edge does
    gen = _generator()
    with open(gen.HEADER_PATH) as f:
        assert f.read() == gen.header_text(), "run `python tools/gen_mc_tables.py` to regenerate csrc/mc_tables.h"
    # the oracle's data file holds the generator's numbers too (and the same geometry conventions)
    assert np.array_equal(mc_tables.MC_NTRI, gen.MC_NTRI) and np.array_equal(mc_tables.MC_TRI, gen.MC_TRI)
    assert np.array_equal(mc_tables.EDGES, gen.EDGES) and np.array_equal(mc_tables.CORNERS, gen.CORNERS)


def test_oracle_sphere_area_orientation_and_watertightness():
    res, r = 48, 0.6
    tris = oracle.marching_cubes(_sphere(res, r))
    area = np.linalg.norm(np.cross(tris[:, 1] - tris[:, 0], tris[:, 2] - tris[:, 0]), axis=1).sum() / 2
    assert abs(area / (4 * np.pi * r * r) - 1) < 5e-3
    n = np.cross(tris[:, 1] - tris[:, 0], tris[:, 2] - tris[:, 0])
    cen = tris.mean(axis=1) - np.array([0.05, -0.1, 0.02], np.float32)
    assert ((n * cen).sum(1) > 0).all()                       # normals point outward (towards sdf > 0)
    assert oracle.mesh_is_closed(tris)
    # every ambiguous configuration: a random field inside a positive shell still gives a closed, consistently oriented mesh
    rs = np.random.RandomState(0)
    g = np.ones((14, 15, 16), np.float32)
    g[1:-1, 1:-1, 1:-1] = rs.standard_normal((12, 13, 14))
    assert oracle.mesh_is_closed(oracle.marching_cubes(g, res=16))
    assert oracle.marching_cubes(np.ones((4, 4, 4), np.float32)).shape == (0, 3, 3)


def test_every_case_is_oriented_along_the_trilinear_field():
    """Per case, independent of how the tables were generated: with corner values -1 (inside) / +1 (outside) and vertices at
    the edge midpoints, every triangle's normal points along INCREASING trilinear interpolant of the corner values (from
    inside to outside) - 820 triangles over the 254 non-trivial cases."""
    corners = mc_tables.CORNERS.astype(np.float64)

    def trilinear(p, vals):
        x, y, z = p
        w = [(x if c[0] else 1 - x) * (y if c[1] else 1 - y) * (z if c[2] else 1 - z) for c in mc_tables.CORNERS]
        return float(np.dot(w, vals))

    total = 0
    for case in range(1, 255):
        vals = np.array([-1.0 if (case >> i) & 1 else 1.0 for i in range(8)])
        for t in range(int(mc_tables.MC_NTRI[case])):
            es = mc_tables.MC_TRI[case, 3 * t: 3 * t + 3]
            pts = np.array([(corners[mc_tables.EDGES[e, 0]] + corners[mc_tables.EDGES[e, 1]]) / 2 for e in es])
            n = np.cross(pts[1] - pts[0], pts[2] - pts[0])
            assert np.linalg.norm(n) > 1e-9, (case, t)                    # no degenerate triangle in the tables
            n /= np.linalg.norm(n)
            c = pts.mean(axis=0)
            assert trilinear(c + 0.05 * n, vals) > trilinear(c - 0.05 * n, vals), (case, t)
            total += 1
    assert total == int(mc_tables.MC_NTRI.sum()) == 820


def _mesh_volume(tris):
    """Signed volume enclosed by an oriented closed triangle soup (divergence theorem), float64."""
    t = tris.astype(np.float64)
    return float(np.einsum("ij,ij->i", t[:, 0], np.cross(t[:, 1], t[:, 2])).sum() / 6.0)


def _euler_characteristic(tris):
    v = np.ascontiguousarray(tris, dtype=np.float32).reshape(-1, 3)
    _, idx = np.unique(v.view(np.uint32).reshape(-1, 3), axis=0, return_inverse=True)
    f = idx.reshape(-1, 3)
    f = f[(f[:, 0] != f[:, 1]) & (f[:, 1] != f[:, 2]) & (f[:, 0] != f[:, 2])]
    e = np.unique(np.sort(np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]), axis=1), axis=0)
    return int(np.unique(f).size - e.shape[0] + f.shape[0])


def test_tables_against_analytic_shapes():
    """A check of the generated case tables that does not go through the generator's own reasoning: meshes of shapes with
    known volume, area and genus.  A wrong or mis-oriented table entry changes the enclosed volume (divergence theorem over
    the oriented soup), the Euler characteristic or the watertightness of at least one of them; the offsets and radii are
    irrational-ish so that the cells see many different sign configurations, ambiguous faces included (the two tori touch
    cells diagonally)."""
    res = 56
    a = oracle.axis_coords(res)
    zz, yy, xx = np.meshgrid(a, a, a, indexing="ij")
    # ellipsoid x^2/a^2 + y^2/b^2 + z^2/c^2 = 1 as the level set of a smooth function (not a distance, which is fine)
    ea, eb, ec = 0.71, 0.52, 0.43
    f = (np.sqrt(((xx - 0.031) / ea) ** 2 + ((yy + 0.017) / eb) ** 2 + ((zz - 0.023) / ec) ** 2) - 1.0).astype(np.float32)
    t = oracle.marching_cubes(f)
    assert oracle.mesh_is_closed(t) and _euler_characteristic(t) == 2
    assert abs(_mesh_volume(t) / (4.0 / 3.0 * np.pi * ea * eb * ec) - 1) < 1e-2
    # torus (genus 1): R = 0.55, r = 0.21, axis z, centre offset
    R, r = 0.55, 0.21
    q = np.sqrt((xx - 0.013) ** 2 + (yy + 0.029) ** 2) - R
    g = (np.sqrt(q ** 2 + (zz - 0.041) ** 2) - r).astype(np.float32)
    t = oracle.marching_cubes(g)
    assert oracle.mesh_is_closed(t) and _euler_characteristic(t) == 0
    assert abs(_mesh_volume(t) / (2 * np.pi ** 2 * R * r * r) - 1) < 1e-2
    area = np.linalg.norm(np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0]), axis=1).sum() / 2
    assert abs(area / (4 * np.pi ** 2 * R * r) - 1) < 1e-2
    # the complement: an inside-out field (everything inside except a ball) bounded by a positive shell; volume = box - ball
    h = -_sphere(res, 0.5)
    h[0], h[-1], h[:, 0], h[:, -1], h[:, :, 0], h[:, :, -1] = 1, 1, 1, 1, 1, 1
    t = oracle.marching_cubes(h)
    assert oracle.mesh_is_closed(t) and _euler_characteristic(t) == 4            # two spheres' worth: the shell and the cavity
    box = (a[-2] - a[1] + (a[1] - a[0])) ** 3                                   # roughly the shell's extent; only the sign matters here
    assert 0 < _mesh_volume(t) < box
    # two unions of shapes -> components add up
    u = np.minimum(_sphere(res, 0.3, (-0.45, -0.4, -0.42)), _sphere(res, 0.33, (0.43, 0.41, 0.4)))
    t = oracle.marching_cubes(u)
    assert oracle.mesh_is_closed(t) and _euler_characteristic(t) == 4
    assert abs(_mesh_volume(t) / (4.0 / 3.0 * np.pi * (0.3 ** 3 + 0.33 ** 3)) - 1) < 2e-2


@pytest.mark.gpu
def test_cuda_marching_cubes_bit_exact(pkg, cuda_decoder):
    rs = np.random.RandomState(3)
    fields = [(_sphere(40), 40, 0), (rs.standard_normal((9, 13, 13)).astype(np.float32), 13, 2),
              (rs.standard_normal((33, 35, 35)).astype(np.float32), 35, 0), (np.ones((5, 6, 6), np.float32), 6, 0)]
    for f, res, z0 in fields:
        got = pkg.extract_surface(torch.from_numpy(f).cuda(), res=res, z0=z0).cpu().numpy()
        want = oracle.marching_cubes(f, res=res, z0=z0)
        assert got.shape == want.shape
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # decoded shape: the decoder's own sign bit-planes drive the classification
    z = oracle.default_latent()
    tris = cuda_decoder.extract_surface(z, 64).cpu().numpy()
    sdf = cuda_decoder.decode_grid(z, 64).cpu().numpy()
    want = oracle.marching_cubes(sdf)
    assert np.array_equal(tris.view(np.uint32), want.view(np.uint32))
    assert tris.shape[0] > 10000
    # a z-slab placed in the grid: same triangles as the corresponding cells of the full extraction
    slab, signs, _ = cuda_decoder.decode_grid_bits(z, 64, 16, 25, mask=False)
    part = pkg.extract_surface(slab, res=64, z0=16, sign_words=signs).cpu().numpy()
    assert np.array_equal(part.view(np.uint32), oracle.marching_cubes(sdf[16:25], res=64, z0=16).view(np.uint32))


@pytest.mark.gpu
def test_cuda_marching_cubes_full_size(pkg, cuda_decoder):
    """256^3 (BASELINE configs[1]'s grid): finite, inside the cube, and a 20-plane slab of it bit-exact with the oracle."""
    z = oracle.default_latent()
    sdf, signs, _ = cuda_decoder.decode_grid_bits(z, 256, mask=False)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    tris = pkg.extract_surface(sdf, 256, 0, sign_words=signs)
    b.record()
    b.synchronize()
    print(f"256^3 marching cubes: {tris.shape[0]} triangles in {a.elapsed_time(b):.2f} ms")
    assert tris.shape[0] > 200000 and torch.isfinite(tris).all() and tris.abs().max() <= 1.0
    slab = sdf[100:120].contiguous()
    part = pkg.extract_surface(slab, 256, 100).cpu().numpy()
    want = oracle.marching_cubes(slab.cpu().numpy(), res=256, z0=100)
    assert np.array_equal(part.view(np.uint32), want.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("res,seed,scale", [(64, 0, 1.0), (97, 1, 1.0), (130, 2, 1.0), (256, 0, 1.0), (256, 3, 1.5), (255, 5, 0.5), (512, 0, 1.0)])
def test_hierarchical_sparse_extraction_equals_dense(cuda_decoder, res, seed, scale):
    """The two-level sparse decode (corners of 8^3 blocks -> lattice of 2^3 sub-blocks -> remaining nodes, every node once)
    followed by the DENSE marching-cubes kernels gives the dense extraction's triangle soup bit for bit, ORDER INCLUDED, and
    the complete sign bit-planes it builds (decoded signs + inherited signs of the discarded regions) equal the dense ones.
    Different latents and latent scales vary the shapes; odd sizes make every level ragged at the upper faces."""
    z = oracle.default_latent(seed) * np.float32(scale)
    sdf_d, signs_d, _ = cuda_decoder.decode_grid_bits(z, res, mask=False)
    dense = cuda_decoder.extract_surface(z, res)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cuda_decoder.extract_surface_sparse(z, res)
    a.record()
    sparse, st = cuda_decoder.extract_surface_sparse(z, res, return_stats=True)
    b.record()
    b.synchronize()
    print(f"res {res} latent {seed} x{scale}: {st['queries']} of {st['dense_queries']} queries ({st['dense_queries'] / max(st['queries'], 1):.1f}x fewer: "
          f"{st['corner_queries']} corners, {st['blocks_kept']} blocks -> {st['lattice_queries']} lattice nodes, {st['sub_blocks_kept']} sub-blocks -> "
          f"{st['fill_queries']} more), {sparse.shape[0]} triangles in {a.elapsed_time(b):.2f} ms, L1 {st['lipschitz_level1']:.2f} L2 {st['lipschitz_level2']:.2f}")
    assert sparse.shape == dense.shape and torch.equal(sparse, dense)
    assert dense.shape[0] > 1000                                                 # a real surface (not a saturated field)
    sdf_s, signs_s, _ = cuda_decoder.decode_sparse_field(z, res)
    nw = (res ** 3 + 31) // 32
    assert torch.equal(signs_s[:nw], signs_d[:nw])                               # every node's sign, decoded or inherited
    act = cuda_decoder.decode_grid(z, res, mask=True)[1].bool()                  # cells the surface crosses: all 8 corners were decoded
    for dz in (0, 1):
        for dy in (0, 1):
            for dx in (0, 1):
                va = sdf_s[dz:res - 1 + dz, dy:res - 1 + dy, dx:res - 1 + dx][act]
                vb = sdf_d[dz:res - 1 + dz, dy:res - 1 + dy, dx:res - 1 + dx][act]
                assert torch.equal(va, vb)
    if res >= 256 and scale == 1.0:
        assert st["queries"] < st["dense_queries"] * (0.2 if res >= 512 else 0.4)


@pytest.mark.gpu
@pytest.mark.parametrize("res,seed,scale", [(128, 0, 1.0), (256, 0, 1.0), (256, 3, 1.5), (255, 5, 0.5), (512, 0, 1.0), (512, 2, 1.0)])
def test_hierarchical_sparse_local_slopes_equal_dense(cuda_decoder, res, seed, scale):
    """local_floor = 0.5: level 2 uses every 8^3 block's own largest difference quotient (x 1.25, never below half the global
    one) instead of the global maximum - a thinner band.  Still the dense extraction's soup, bit for bit, on every test shape."""
    z = oracle.default_latent(seed) * np.float32(scale)
    dense = cuda_decoder.extract_surface(z, res)
    cuda_decoder.extract_surface_sparse(z, res, local_floor=0.5)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    sparse, st = cuda_decoder.extract_surface_sparse(z, res, local_floor=0.5, return_stats=True)
    b.record()
    b.synchronize()
    _, st_g = cuda_decoder.extract_surface_sparse(z, res, return_stats=True)
    print(f"res {res} latent {seed} x{scale}: local slopes {st['queries']} queries ({st['dense_queries'] / max(st['queries'], 1):.1f}x fewer) in "
          f"{a.elapsed_time(b):.2f} ms; global bound {st_g['queries']} queries; {sparse.shape[0]} triangles")
    assert sparse.shape == dense.shape and torch.equal(sparse, dense)
    assert st["queries"] <= st_g["queries"]


@pytest.mark.gpu
def test_indexed_mesh_welding(pkg, cuda_decoder):
    """indexed=True merges vertices by grid edge: the faces index exactly the soup's vertices, a closed surface
    has Euler characteristic 2, and the sparse extractor welds to the same mesh."""
    f = torch.from_numpy(_sphere(40)).cuda()
    soup = pkg.extract_surface(f)
    verts, faces = pkg.extract_surface(f, indexed=True)
    assert faces.shape == (soup.shape[0], 3) and faces.dtype == torch.int64
    assert torch.equal(verts[faces], soup)                                   # same geometry, bit for bit
    uniq = np.unique(soup.cpu().numpy().reshape(-1, 3).view(np.uint32), axis=0).shape[0]
    assert verts.shape[0] == uniq                                            # one vertex per crossed edge
    fa = faces.cpu().numpy()
    e = np.sort(np.concatenate([fa[:, [0, 1]], fa[:, [1, 2]], fa[:, [2, 0]]]), axis=1)
    n_edges = np.unique(e, axis=0).shape[0]
    assert verts.shape[0] - n_edges + fa.shape[0] == 2                       # a sphere
    z = oracle.default_latent()
    v1, f1 = cuda_decoder.extract_surface(z, 97, indexed=True)
    v2, f2 = cuda_decoder.extract_surface_sparse(z, 97, indexed=True)         # same soup, same order
    assert torch.equal(v1, v2) and torch.equal(f1, f2)


@pytest.mark.gpu
@pytest.mark.parametrize("res", [65, 96])
@pytest.mark.parametrize("width_cells", [0.8, 1.5])
def test_sparse_extraction_keeps_a_thin_slab(pkg, res, width_cells):
    """A feature thinner than a block that no block corner sees: a decoder whose field is exactly tanh(|n.x - d| - half),
    n = (0.5, 0.5, 0.5) - 1-Lipschitz, negative only inside a planar slab `width_cells` cells wide, with d between the planes
    of level-1 corners.  Layer 0 forms n.x - d and d - n.x (exact bf16 weights), layers 1-7 pass those two channels through
    with identity weights, the head adds them.  With the bound L = 1 the two-level decode keeps every block and sub-block the
    slab crosses and the nodes it never decodes inherit the right sign: the soup equals the dense extraction's bit for bit,
    order included."""
    from oracle.weights import DEC_LAYER_DIMS
    h = 2.0 / (res - 1)
    # n.x at node (i, j, k) is -1.5 + h (i + j + k) / 2: level-1 corners (multiples of 8) lie on the planes n.x = -1.5 + 4h M
    d = -1.5 + h * (4 * int(0.75 * (res - 1) / 4) + 2.45)
    half = 0.5 * width_cells * h * np.sqrt(0.75)                                # |n| = sqrt(3) / 2
    params = [(np.zeros((fout, fin), np.float32), np.zeros(fout, np.float32)) for fin, fout in DEC_LAYER_DIMS]
    (w0, b0), (w8, b8) = params[0], params[8]
    w0[0, 256:], b0[0] = 0.5, -d
    w0[1, 256:], b0[1] = -0.5, d
    for w, _ in params[1:8]:                                                    # layer 4: columns 0, 1 of [h3 | latent | xyz]
        w[0, 0] = w[1, 1] = 1.0
    w8[0, :2], b8[0] = 1.0, -half
    a = oracle.axis_coords(res).astype(np.float64)[np.minimum(np.arange(0, res + 7, 8), res - 1)]
    cz, cy, cx = np.meshgrid(a, a, a, indexing="ij")
    assert not (np.abs(0.5 * (cx + cy + cz) - d) < half).any()                 # no level-1 corner is inside the slab
    z = np.zeros(256, np.float32)
    dec = pkg.Decoder(params, device="cuda:0", precision="bf16")
    try:
        dense = dec.extract_surface(z, res)
        sparse, st = dec.extract_surface_sparse(z, res, lipschitz=1.0, return_stats=True)
    finally:
        dec.close()
    print(f"res {res}, slab of {width_cells} cells: {st['queries']} of {st['dense_queries']} queries ({st['corner_queries']} corners, "
          f"{st['blocks_kept']} blocks, {st['lattice_queries']} lattice nodes, {st['sub_blocks_kept']} sub-blocks, {st['fill_queries']} more), "
          f"{sparse.shape[0]} triangles")
    assert dense.shape[0] > 1000
    assert sparse.shape == dense.shape and torch.equal(sparse, dense)
    assert st["queries"] < st["dense_queries"]
