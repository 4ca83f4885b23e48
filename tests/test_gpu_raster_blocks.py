"""k_raster's two warp-block heights (csrc/nr_raster.cu) against the oracle.

A warp of k_raster owns an 8x8 pixel block (two pixels per lane, the lower one four rows below the upper)
when there is a lot of work, and an 8x4 block (the upper half only) when even the 8x4 blocks of all non-empty
tiles fit in one wave of resident warps.  The kernel picks the height from the number of non-empty tiles
(nr_raster.cu:138), so small test inputs only ever run 8x4 blocks.  Views are independent, so these tests reach
8x8 blocks by rendering a case's views many times over in one call (the oracle runs once per original view and
every copy is compared with it), and 8x4 blocks by rendering the case as it is.  `copies` chooses the number of
copies and asserts that the call really runs the height asked for: a lower bound on the non-empty tiles (the
tiles holding a covered pixel of the oracle's face_index_map) of at least twice the threshold for 8x8 blocks,
the upper bound B * tiles per view for 8x4 blocks.  If the threshold moves, these tests fail instead of
quietly testing one height.

Bars: face_index_map and weight_map bit-exact, images within rtol 1e-5, atol 1e-6 of the reference and
bit-identical between the 8x4 and the 8x8 run of the same view (the per-pixel arithmetic is the same),
gradients within test_gpu_parity.py's bar."""
import ctypes
import os

import numpy as np
import pytest
import torch

import oracle
from oracle import pipeline as ref
from test_gpu_parity import CASES, GOLDEN, _check_vs_oracle, grad_close, random_triangles, run_cuda
import test_gpu_light_gradients as lg
import test_gpu_reference_kernels as rk

pytestmark = pytest.mark.gpu

RASTER_WARPS = 8            # TILE_THREADS / 32 (nr_raster.cu:68)
SHARED = ("faces", "faces_textures")        # fixture arrays that are not per view


@pytest.fixture(scope="module")
def nr():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import neural_renderer_v2_pytorch_b200 as nr_
    return nr_


def block_threshold(fine):
    """The most non-empty tiles at which k_raster still runs 8x4 blocks: it runs 8x8 blocks iff
    tiles * (FINE ? 2 : 8) > sm_count * 4 * RASTER_WARPS (nr_raster.cu:138; sm_count is sm_count_cached(),
    the device's multiprocessor count)."""
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    return sm * 4 * RASTER_WARPS // (2 if fine else 8)


def covered_tiles(fim, tile):
    """Tiles of fim [B, R, R] holding a covered pixel: each has a non-empty face list."""
    B, R = fim.shape[:2]
    n = -(-R // tile)
    p = np.full((B, n * tile, n * tile), -1, np.int64)
    p[:, :R, :R] = fim
    return int((p.reshape(B, n, tile, n, tile) >= 0).any(axis=(2, 4)).sum())


def copies(fim, height, fine=None):
    """How many times to render the views whose face_index_map is fim [B, R, R] so that k_raster runs
    `height` ("8x8" or "8x4") blocks, on 16x16 tiles (fine False), 8x8 tiles (fine True) or both (None)."""
    B, R = fim.shape[:2]
    k = 1
    for f in ((False, True) if fine is None else (fine,)):
        t, tile = block_threshold(f), 8 if f else 16
        if height == "8x4":
            ntx = -(-R // tile)
            assert B * ntx * ntx <= t, "%d tiles can run 8x8 blocks (threshold %d)" % (B * ntx * ntx, t)
        else:
            assert height == "8x8", height
            n = covered_tiles(fim, tile)
            assert n > 0, "nothing covered"
            k = max(k, -(-2 * t // n))
    if height == "8x8":
        for f in ((False, True) if fine is None else (fine,)):
            t, tile = block_threshold(f), 8 if f else 16
            assert k * covered_tiles(fim, tile) >= 2 * t
    return k


def at_block(case, height, fim, fine=None):
    """The fixture dict `case` with every per-view array (inputs, expected outputs, gradients) repeated
    copies(fim, height, fine) times along the view axis -> (dict, copies)."""
    B = fim.shape[0]
    k = copies(fim, height, fine)
    out = {key: np.concatenate([v] * k) if key not in SHARED and np.ndim(v) and len(v) == B else v
           for key, v in case.items()}
    return out, k


def fixture(name):
    d = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    if "face_index_map" in d:
        return d, d["face_index_map"]
    R = int(d["image_size"]) * (2 if bool(d["anti_aliasing"]) else 1)
    f = np.ascontiguousarray(d["vertices"][:, d["faces"]], dtype=np.float32)
    return d, oracle.face_index_map(f, R, float(d["near"]), float(d["far"]), bool(d["draw_backside"]))


def check_fixture(d, images, v, tex, vt, maps):
    """test_gpu_parity.py::test_golden_case's bars, on every copy."""
    if "face_index_map" in d:
        assert np.array_equal(maps["face_index_map"].cpu().numpy(), d["face_index_map"]), "face_index_map not bit-exact"
        assert np.array_equal(maps["weight_map"].cpu().numpy(), d["weight_map"]), "weight_map differs"
    np.testing.assert_allclose(images.detach().cpu().numpy(), d["images"], rtol=1e-5, atol=1e-6)
    grad_close(v.grad.cpu().numpy(), d["grad_vertices"], "grad_vertices")
    if tex is not None:
        grad_close(tex.grad.cpu().numpy(), d["grad_textures"], "grad_textures")
        grad_close(vt.grad.cpu().numpy(), d["grad_vertices_textures"], "grad_vertices_textures")


def same_per_copy(t, B, what):
    """Every copy of a [k * B, ...] result equals copy 0, bit for bit."""
    t = t.detach().reshape((-1, B) + tuple(t.shape[1:]))
    for j in range(1, t.shape[0]):
        assert torch.equal(t[j], t[0]), "%s: copy %d differs from copy 0" % (what, j)


class _Hooks:
    """rasterize.py's path switches, set for the duration of a run."""

    def __init__(self, **kw):
        self.kw = kw

    def __enter__(self):
        from neural_renderer_v2_pytorch_b200 import rasterize as rz
        self.rz, self.saved = rz, {k: getattr(rz, k) for k in self.kw}
        for k, v in self.kw.items():
            setattr(rz, k, v)

    def __exit__(self, *exc):
        for k, v in self.saved.items():
            setattr(self.rz, k, v)


def both_heights(nr, name, fine=False, **hooks):
    """Fixture `name` at 8x4 and at 8x8 blocks: every bar on every copy, and the 8x8 images of every copy equal
    to the 8x4 images bit for bit.  -> the 8x8 run's (images, v, tex, vt, maps, copies)."""
    d, fim = fixture(name)
    runs = {}
    for height in ("8x4", "8x8"):
        p, k = at_block(d, height, fim, fine)
        with _Hooks(FORCE_FINE_TILES=fine, **hooks):
            out = run_cuda(nr, p)
        check_fixture(p, *out)
        runs[height] = out + (k,)
    B = fim.shape[0]
    img4, img8 = runs["8x4"][0].detach(), runs["8x8"][0].detach()
    assert torch.equal(img8.reshape((-1,) + tuple(img4.shape))[0], img4)
    same_per_copy(img8, B, "images")
    return runs["8x8"]


# ------------------------------------------------------------------------------------------- fixtures

@pytest.mark.parametrize("name", CASES)
def test_golden_case_at_both_heights(nr, name):
    both_heights(nr, name)


@pytest.mark.parametrize("name", ["case_rgba_64", "case_rgba_aa_32", "case_depth_aa_32", "case_sil_cull_64"])
def test_golden_case_fine_tiles_at_both_heights(nr, name):
    both_heights(nr, name, fine=True)


def test_pair_list_overflow_at_both_heights(nr):
    """No room for the (tile, face) pairs: every block scans every face of its view."""
    both_heights(nr, "case_rgba_64", FORCE_PAIR_CAPACITY=0)


def test_deterministic_mode_at_8x8(nr):
    """Deterministic mode: every copy of a view gets the same gradient bits."""
    images, v, tex, vt, maps, k = both_heights(nr, "case_rgba_64", DETERMINISTIC=True)
    assert k > 1
    B = v.shape[0] // k
    for t, what in ((v.grad, "grad_vertices"), (tex.grad, "grad_textures"), (vt.grad, "grad_vertices_textures")):
        same_per_copy(t, B, what)


@pytest.mark.parametrize("name", lg.FIXTURES)
def test_lights_at_both_heights(nr, name):
    """Directional + ambient + specular lights, every light tensor requiring grad: images and the image and light
    gradients against the fixture and autograd of the oracle (test_gpu_light_gradients.py's bars)."""
    d, fim = fixture(name)
    lb = bool(d["light_backside"])
    want_lights = lg.oracle_grads(name, lb)
    imgs = {}
    for height in ("8x4", "8x8"):
        p, k = at_block(d, height, fim)
        with lg._Mode("tiles"):
            P = lg._light_params(p, "cuda:0", True)
            img, v, tex = lg.render(nr, p, lg._lights(nr, P, lb))
        np.testing.assert_allclose(img.cpu().numpy(), p["images"], rtol=1e-5, atol=2e-6)
        grad_close(tex.grad.cpu().numpy(), p["grad_textures"], "grad_textures")
        gv, want = v.grad.cpu().numpy(), p["grad_vertices"]
        assert np.abs(gv - want).max() <= 1e-4 * np.abs(want).max()
        for key in lg.LIGHT_KEYS:
            grad_close(P[key].grad.cpu().numpy(), np.concatenate([want_lights[key]] * k), key)
        imgs[height] = img
    assert torch.equal(imgs["8x8"].reshape((-1,) + tuple(imgs["8x4"].shape))[0], imgs["8x4"])
    same_per_copy(imgs["8x8"], fim.shape[0], "images")


def teapot_views(nr, B, seed):
    d = np.load(os.path.join(GOLDEN, "teapot.npz"))
    g = torch.Generator().manual_seed(seed)
    vw = torch.from_numpy(d["vertices"])[None].repeat(B, 1, 1)
    eye = nr.get_points_from_angles(torch.full((B,), 2.732), torch.rand(B, generator=g) * 80 - 20,
                                    torch.rand(B, generator=g) * 360)
    return nr.perspective(nr.look_at(vw, eye)), torch.from_numpy(d["faces"]), g


@pytest.mark.parametrize("aa,mode", [(False, "picture"), (True, "picture"), (True, "color")])
def test_backgrounds_at_8x8(nr, aa, mode):
    """test_gpu_parity.py::test_backgrounds with every view repeated: images and the gradients to vertices,
    textures and the background picture against the oracle."""
    B, S, ts = 2, 48, 2
    R = 2 * S if aa else S
    vs, faces, g = teapot_views(nr, B, 7)
    vt_np, ft_np, tex_np = nr.create_textures(faces.shape[0], ts)
    tex0 = torch.rand((B,) + tex_np.shape, generator=g)
    vt0 = torch.from_numpy(vt_np)[None].repeat(B, 1, 1)
    G = torch.randn((B, 4, S, S), generator=g)
    color = [0.25, 0.5, 0.75]
    bg0 = torch.rand((B, 3, R, R), generator=g) if mode == "picture" else \
        torch.tensor(color)[None, :, None, None].expand(B, 3, R, R).contiguous()
    v0, t0, b0 = (x.clone().requires_grad_(True) for x in (vs, tex0, bg0))
    img0, maps0 = ref.rasterize(v0, faces, S, aa, draw_rgb=True, draw_silhouettes=True, vertices_textures=vt0,
                                faces_textures=ft_np, textures=t0, backgrounds=b0, return_maps=True)
    (img0 * G).sum().backward()
    k = copies(maps0["face_index_map"].numpy(), "8x8", False)
    rep = lambda x: torch.cat([x.detach()] * k).cuda()
    v1, t1, b1 = (rep(x).requires_grad_(True) for x in (vs, tex0, bg0))
    kw = dict(backgrounds=b1) if mode == "picture" else dict(background_color=color)
    p = nr.RasterizeParam(vertices_textures=rep(vt0), faces_textures=torch.from_numpy(ft_np).cuda(), textures=t1, **kw)
    img1 = nr.rasterize_rgba(v1, faces.cuda(), p, nr.RasterizeHyperparam(image_size=S, anti_aliasing=aa))
    (img1 * rep(G)).sum().backward()
    tile = lambda x: np.concatenate([x.detach().numpy()] * k)
    np.testing.assert_allclose(img1.detach().cpu().numpy(), tile(img0), rtol=1e-5, atol=1e-6)
    grad_close(v1.grad.cpu().numpy(), tile(v0.grad), "grad_vertices")
    grad_close(t1.grad.cpu().numpy(), tile(t0.grad), "grad_textures")
    if mode == "picture":
        grad_close(b1.grad.cpu().numpy(), tile(b0.grad), "grad_backgrounds")


# ------------------------------------------------------------------------- geometry aimed at the halves

def ndc(p, R):
    """pixel coordinate (pixel centres at integers) -> screen coordinate, pix_center (nr_common.cuh:90)"""
    return (2. * np.asarray(p, np.float64) + 1 - R) / R


def tri(x0, y0, x1, y1, x2, y2, z, R):
    """one face from pixel coordinates, corner depths z (scalar or 3)"""
    xy = np.array([[x0, y0], [x1, y1], [x2, y2]], np.float64)
    zz = np.broadcast_to(np.asarray(z, np.float64), (3,))
    return np.concatenate([ndc(xy, R), zz[:, None]], 1)


def check_heights(nr, faces, R, **kw):
    """_check_vs_oracle at 8x4 and at 8x8 blocks: the reference-signature operators and the fused forward on
    16x16 tiles (one-kernel and general binning) and on 8x8 tiles."""
    faces = np.ascontiguousarray(faces, dtype=np.float32)
    for height in ("8x4", "8x8"):
        _check_vs_oracle(nr, faces, R, copies=lambda fim: copies(fim, height), **kw)


def box_faces(R, boxes):
    """Block i of the view (raster order) gets two faces whose exact pixel box is columns c0..c1 and rows r0..r1
    of the block (vertex extents end between a quarter and a half pixel beyond the outer pixel centres), under a
    full-screen face at depth 5 that every block lists."""
    nb = R // 8
    out = [tri(-2 * R, -2 * R, 5 * R, -2 * R, -2 * R, 5 * R, 5.0, R)]
    for i, (c0, c1, r0, r1) in enumerate(boxes):
        bx, by = (i % nb) * 8, (i // nb) * 8
        z = 1.0 + 0.01 * (i % 7)
        out.append(tri(bx + c0 - .25, by + r0 - .25, bx + c1 + .45, by + r0 - .25, bx + c0 - .25, by + r1 + .45, z, R))
        out.append(tri(bx + c1 + .25, by + r1 + .25, bx + c1 + .25, by + r0 - .45, bx + c0 - .45, by + r1 + .25, z + 3e-3, R))
    return out


def test_pixel_boxes_at_every_row_range(nr):
    """Faces whose pixel boxes cover every row range 0 <= r0 <= r1 <= 7 of a block against several column ranges:
    boxes in the upper half only, in the lower half only (upper mask word 0), straddling rows 3|4, on row 7 alone."""
    R = 64
    boxes = [(c0, c1, r0, r1) for r0 in range(8) for r1 in range(r0, 8)
             for c0, c1 in ((0, 7), (0, 0), (7, 7), (2, 5), (3, 4))]
    per_view = (R // 8) ** 2
    views = [box_faces(R, boxes[v:v + per_view]) for v in range(0, len(boxes), per_view)]
    nf = max(len(f) for f in views)
    pad = tri(3 * R, 3 * R, 3 * R + 1, 3 * R, 3 * R, 3 * R + 1, 1.0, R)        # off screen
    faces = np.stack([np.stack(f + [pad] * (nf - len(f))) for f in views])
    check_heights(nr, faces, R)


def test_single_pixel_faces_at_every_block_position(nr):
    """One face per block covering only the pixel centre at (c, r) of that block, for all 64 positions."""
    R = 64
    faces = np.stack(box_faces(R, [(c, c, r, r) for r in range(8) for c in range(8)]))[None]
    check_heights(nr, faces, R)


def test_edges_through_pixel_centres_on_block_rows(nr):
    """test_gpu_parity.py::test_vertices_on_pixel_centres with the v1-v2 edge on block rows / columns 3, 4 (the
    halves' boundary), 7 and 8 (the blocks' boundary): the c2 == 0 pixels there must survive both culls."""
    R = 64
    rng = np.random.RandomState(34)
    for size in (5, 14):
        centre = rng.randint(0, R, size=(2, 600, 1, 2))
        px = np.clip(centre + rng.randint(-size, size + 1, size=(2, 600, 3, 2)), -8, R + 8).astype(np.float64)
        line = 8 * rng.randint(0, R // 8, size=(2, 600)) + rng.choice([3, 4, 7, 8], size=(2, 600))
        px[:, :200, 1, 1] = px[:, :200, 2, 1] = line[:, :200]        # horizontal edge v1-v2 on a pixel row
        px[:, 200:400, 1, 0] = px[:, 200:400, 2, 0] = line[:, 200:400]   # vertical edge on a pixel column
        z = rng.uniform(1., 3., size=(2, 600, 3, 1))
        f = np.concatenate([ndc(px, R), z], -1)
        check_heights(nr, f, R)
        check_heights(nr, f, R, backside=False)


def test_multi_group_lists_alternating_halves(nr):
    """96 faces per block, in three groups of 32 list entries whose survivors all lie in one half (lower, upper,
    lower or the reverse): the z state of both pixels is carried across groups that skip it."""
    R = 64
    rng = np.random.RandomState(5)
    views = []
    for v in range(2):
        f = []
        for blk in range((R // 8) ** 2):
            bx, by = (blk % 8) * 8, (blk // 8) * 8
            for grp in range(3):
                lower = (grp + blk + v) % 2 == 0
                for _ in range(32):
                    x = bx + rng.uniform(-.4, 7.4, 3)
                    y = by + (4 if lower else 0) + rng.uniform(-.4, 3.4, 3)
                    f.append(tri(x[0], y[0], x[1], y[1], x[2], y[2], rng.uniform(1., 3., 3), R))
        views.append(np.stack(f))
    check_heights(nr, np.stack(views), R)


def test_hysteresis_stacks_in_the_lower_half(nr):
    """test_gpu_parity.py::test_hysteresis_is_order_dependent's stacks of three faces 5e-5 .. 2e-4 apart in
    depth, placed in rows 4..7 of every block and tilted in y (depth changes by 1e-2 over four rows): the
    near-tie fallback of the lower pixel recomputes the winner's depth at that pixel's own row."""
    R = 64
    stacks = ([1.0, 0.99995, 0.9999], [0.9999, 0.99995, 1.0], [1.0, 0.9998, 0.99975])
    views = []
    for slope in (2.5e-3, -2.5e-3):     # depth per pixel row
        f = []
        for blk in range((R // 8) ** 2):
            bx, by = (blk % 8) * 8, (blk // 8) * 8
            for z in stacks[blk % 3]:
                ys = np.array([by + 3.6, by + 3.6, by + 7.4])
                f.append(tri(bx - .4, ys[0], bx + 7.4, ys[1], bx + 3.5, ys[2], z + slope * (ys - by - 4), R))
        views.append(np.stack(f))
    check_heights(nr, np.stack(views), R)


@pytest.mark.parametrize("name", ["ties_300_0.0002", "ties_5000_0.0003", "ties_5000_0.05"])
def test_reference_kernel_ties_at_8x8(nr, name):
    """The piles of near-ties whose reference-kernel output is stored, through the tile pipeline at 8x8 blocks:
    every copy is the reference kernel's map, bit for bit."""
    faces, S, near, far, bs = rk.mk.stress_inputs()[name]
    d = rk.stored(name, faces)
    k = copies(d["face_index_map"], "8x8", False)
    fim, wm = rk.ours(nr, np.concatenate([faces] * k), S, near, far, bs)
    B = faces.shape[0]
    for j in range(k):
        rk.assert_maps(d, fim[j * B:(j + 1) * B], wm[j * B:(j + 1) * B], "tile pipeline, copy %d" % j)


def test_non_finite_vertices_at_both_heights(nr):
    f = random_triangles(1, 400, 4, size=0.3)
    f[0, 3, 0, 0] = np.nan
    f[0, 9, 1, 1] = np.inf
    f[0, 15, 2, 0] = -np.inf
    f[0, 21, 0, 2] = np.nan
    f[0, 27, 1, 2] = np.inf
    f[0, 33, 2, 2] = 0.0
    f[0, 39, :, 2] = -1.0
    check_heights(nr, f, 96)


def test_near_far_clipping_at_both_heights(nr):
    check_heights(nr, random_triangles(2, 2000, 6, size=0.1, zlo=0.05, zhi=4.0), 128, near=1.0, far=2.5)


@pytest.mark.parametrize("S,aa", [(100, False), (104, False), (108, False), (50, True), (52, True)])
@pytest.mark.parametrize("fine", [False, True])
def test_partial_tiles_full_variant(nr, S, aa, fine):
    """Image sizes that are no multiple of 16 (the lower half of a block, or a tile's second block row, lies
    outside the image): the FULL variant with textures, weight map and depth map (rasterize_maps, RGBA and depth
    channels) against oracle/pipeline.py, at both heights."""
    B, ts = 2, 2
    vs, faces, g = teapot_views(nr, B, S)
    vt_np, ft_np, tex_np = nr.create_textures(faces.shape[0], ts)
    tex0 = torch.rand((B,) + tex_np.shape, generator=g)
    vt0 = torch.from_numpy(vt_np)[None].repeat(B, 1, 1)
    img0, maps0 = ref.rasterize(vs, faces, S, aa, draw_rgb=True, draw_silhouettes=True, draw_depth=True,
                                vertices_textures=vt0, faces_textures=ft_np, textures=tex0, return_maps=True)
    fim0, wm0 = maps0["face_index_map"].numpy(), maps0["weight_map"].numpy()
    dm0 = ref.compute_depth_map(vs[:, faces.long()], maps0["face_index_map"], maps0["weight_map"]).numpy()
    imgs = {}
    for height in ("8x4", "8x8"):
        k = copies(fim0, height, fine)
        rep = lambda x: torch.cat([x] * k).cuda()
        hp = nr.RasterizeHyperparam(image_size=S, anti_aliasing=aa, draw_rgb=True, draw_silhouettes=True, draw_depth=True)
        p = nr.RasterizeParam(vertices_textures=rep(vt0), faces_textures=torch.from_numpy(ft_np).cuda(), textures=rep(tex0))
        with _Hooks(FORCE_FINE_TILES=fine):
            maps = nr.rasterize_maps(rep(vs), faces.cuda(), p, hp)
        tile = lambda x: np.concatenate([x] * k)
        assert np.array_equal(maps["face_index_map"].cpu().numpy(), tile(fim0)), "face_index_map"
        assert np.array_equal(maps["weight_map"].cpu().numpy(), tile(wm0)), "weight_map"
        fg = tile(fim0) >= 0
        np.testing.assert_allclose(maps["depth_map"].cpu().numpy()[fg], tile(dm0)[fg], rtol=1e-6)
        np.testing.assert_allclose(maps["images"].cpu().numpy(), tile(img0.numpy()), rtol=1e-5, atol=1e-6)
        imgs[height] = maps["images"]
    assert torch.equal(imgs["8x8"][:B], imgs["8x4"])
    same_per_copy(imgs["8x8"], B, "images")


# ------------------------------------------------------------------------------------ the switch itself

def one_face_per_tile(R, tile, placed, nviews):
    """nviews views at R; the first `placed` tiles (view-major) each get one small face strictly inside them,
    every other face of a view lies off screen.  -> faces [nviews, tiles per view, 3, 3]."""
    nt = R // tile
    off = tri(3 * R, 3 * R, 3 * R + 1, 3 * R, 3 * R, 3 * R + 1, 1.0, R)
    faces = np.empty((nviews, nt * nt, 3, 3))
    for v in range(nviews):
        for t in range(nt * nt):
            i = v * nt * nt + t
            x, y = (t % nt) * tile + tile // 2, (t // nt) * tile + tile // 2
            faces[v, t] = tri(x - 2.3, y - 1.6, x + 1.8, y - 2.2, x - .5, y + 2.1, 1.0 + 1e-3 * t, R) if i < placed else off
    return np.ascontiguousarray(faces, dtype=np.float32)


@pytest.mark.parametrize("fine", [False, True])
def test_block_height_switch(nr, fine):
    """Exactly `threshold` non-empty tiles (8x4 blocks) and threshold + 1 (8x8 blocks).  Every CTA decides the
    height from the tile count for itself; had any CTA decided otherwise, blocks would be missing (poison left in
    the outputs) or doubled.  Every view must be the oracle's, bit for bit."""
    from neural_renderer_v2_pytorch_b200 import _lib
    L = _lib.lib()
    R, tile = 64, (8 if fine else 16)
    t = block_threshold(fine)
    per_view = (R // tile) ** 2
    for placed in (t, t + 1):
        nviews = -(-placed // per_view)
        faces = one_face_per_tile(R, tile, placed, nviews)
        want = oracle.face_index_map(faces, R)
        assert covered_tiles(want, tile) == placed      # each face's pixel box lies inside its tile
        if placed == t:
            assert copies(want, "8x4", fine) == 1
        B, nf = faces.shape[:2]
        v = torch.from_numpy(faces).reshape(B, nf * 3, 3).cuda()
        idx = torch.arange(nf * 3, dtype=torch.int32).reshape(nf, 3).cuda()
        flags = _lib.NR_DRAW_SILHOUETTES | _lib.NR_DRAW_BACKSIDE | (_lib.NR_FINE_TILES if fine else 0)
        cfg = _lib.RasterConfig(batch=B, num_vertices=nf * 3, num_faces=nf, image_size=R, flags=flags, near_plane=0.1,
                                far_plane=100., eps=1e-5, depth_min_delta=1e-4)
        cap = 8 * B * nf
        fim = torch.full((B * R * R,), 0x5a5a5a5a, dtype=torch.int32, device="cuda")
        images = torch.full((B * R * R,), 12345.5, device="cuda")
        tile_list = torch.empty(8 + 16 * B * per_view, dtype=torch.int32, device="cuda")
        ws = torch.empty(int(L.nr_workspace_bytes(ctypes.byref(cfg), cap)) + 256, dtype=torch.uint8, device="cuda")
        base = (ws.data_ptr() + 255) & ~255
        ptr = lambda x: ctypes.c_void_p(x.data_ptr())
        rc = L.nr_rasterize_forward(ctypes.byref(cfg), ptr(v), ptr(idx), None, None, None, ptr(fim), None, None,
                                    ptr(images), None, None, ptr(tile_list), ctypes.c_void_p(base),
                                    ws.numel() - (base - ws.data_ptr()), cap, None, None, None, None,
                                    ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        _lib.check(rc, "forward")
        got = fim.reshape(B, R, R).cpu().numpy()
        assert not (got == 0x5a5a5a5a).any() and not bool((images == 12345.5).any()), "pixels left unwritten"
        assert np.array_equal(got, want), "%d tiles: %d px differ" % (placed, (got != want).sum())
        sil = images.reshape(B, R, R).flip(1, 2).cpu().numpy()
        assert np.array_equal(sil, (want >= 0).astype(np.float32))
