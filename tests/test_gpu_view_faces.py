"""Per-view meshes: faces and faces_textures of shape [B, nf, 3] (NR_VIEW_FACES) through both binning paths, 8x8
tiles, the z-buffer path, both k_raster block heights, the staged and the unstaged backward.

Views are independent, so there are exact bars:
  * the same topology passed as [B, nf, 3] renders what the [nf, 3] call renders: face_index_map, weight map and
    images bit for bit, gradients bit for bit in deterministic mode (fixed-point sums do not depend on the batch) and
    within test_gpu_parity.py's bar with float atomics;
  * a batch of different meshes, padded to common nv / nf (padding faces [0, 0, 0]), renders in every view what a
    single-view call on that view's own unpadded mesh renders."""
import ctypes
import os

import numpy as np
import pytest
import torch

import bench
import oracle
from oracle import pipeline as ref
from test_gpu_parity import CASES, GOLDEN, grad_close, random_triangles
from test_gpu_raster_blocks import _Hooks, at_block, copies, fixture
import test_gpu_light_gradients as lg

pytestmark = pytest.mark.gpu

UNSTAGED = "NR_FORCE_UNSTAGED_BACKWARD"
# rasterize.py's path switches per path name; "8x8" repeats the views until k_raster runs 8x8 blocks
PATHS = {
    "binview": {},
    "general": dict(FORCE_GENERAL_BINNING=True),
    "fine": dict(FORCE_FINE_TILES=True),
    "dense": dict(FORCE_DENSE_RASTER=True),
    "8x8": {},
    "unstaged": {},
    "deterministic": {},
}


@pytest.fixture(scope="module")
def nr():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import neural_renderer_v2_pytorch_b200 as nr_
    return nr_


@pytest.fixture
def unstaged(monkeypatch):
    def set_(on):
        if on:
            monkeypatch.setenv(UNSTAGED, "1")
        else:
            monkeypatch.delenv(UNSTAGED, raising=False)
    return set_


def render(nr, mode, S, aa, v, faces, vt=None, ft=None, tex=None, G=None, lights=None, det=False, backside=True,
           backgrounds=None):
    """One call of the public API: images, maps (face_index_map, weight_map), gradients of every leaf given."""
    hp = nr.RasterizeHyperparam(image_size=S, anti_aliasing=aa, draw_backside=backside)
    hp.deterministic = det
    rgb = mode in ("rgb", "rgba")
    p = nr.RasterizeParam(vertices_textures=vt, faces_textures=ft, textures=tex, lights=lights,
                          backgrounds=backgrounds) if rgb else nr.RasterizeParam()
    fn = {"silhouettes": nr.rasterize_silhouettes, "rgb": nr.rasterize_rgb, "rgba": nr.rasterize_rgba,
          "depth": nr.rasterize_depth}[mode]
    images = fn(v, faces, p, hp)
    if G is not None:
        (images * G[:, 0] if images.ndim == 3 else images * G).sum().backward()
    hp2 = nr.RasterizeHyperparam(image_size=S, anti_aliasing=aa, draw_backside=backside, draw_rgb=rgb,
                                 draw_silhouettes=mode in ("silhouettes", "rgba"), draw_depth=mode == "depth")
    hp2.deterministic = det
    maps = nr.rasterize_maps(v.detach(), faces, p, hp2)
    torch.cuda.synchronize()
    return images.detach(), maps


def leaves(d, dev, keys):
    return {k: torch.from_numpy(np.ascontiguousarray(d[k])).to(dev).requires_grad_(True) for k in keys}


def per_view(t, B):
    return t[None].expand(B, *t.shape).contiguous()


def check_same(a, b, det, what):
    if det:
        assert torch.equal(a, b), "%s: not bit-identical" % what
    else:
        grad_close(a.cpu().numpy(), b.cpu().numpy(), what)


# ---------------------------------------------------------------------------------------------------------------- 1
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("name", CASES)
def test_same_topology_per_view_equals_shared(nr, unstaged, name, path):
    d, fim0 = fixture(name)
    if path == "8x8":
        d, _ = at_block(d, "8x8", fim0)
    mode, S, aa = str(d["mode"]), int(d["image_size"]), bool(d["anti_aliasing"])
    det = path == "deterministic"
    unstaged(path == "unstaged")
    dev = "cuda:0"
    rgb = mode in ("rgb", "rgba")
    B = d["vertices"].shape[0]
    G = torch.from_numpy(d["grad_images"]).to(dev)
    if G.ndim == 3:
        G = G[:, None]
    out = []
    for view_faces in (False, True):
        L = leaves(d, dev, ["vertices"] + (["vertices_textures", "textures"] if rgb else []))
        f = torch.from_numpy(d["faces"]).to(dev)
        ft = torch.from_numpy(d["faces_textures"]).to(dev) if rgb else None
        if view_faces:
            f = per_view(f, B)
            ft = per_view(ft, B) if rgb else None
        with _Hooks(**PATHS[path]):
            images, maps = render(nr, mode, S, aa, L["vertices"], f, L.get("vertices_textures"), ft, L.get("textures"),
                                  G, det=det, backside=bool(d["draw_backside"]))
        out.append((images, maps, L))
    (i0, m0, L0), (i1, m1, L1) = out
    assert torch.equal(m0["face_index_map"], m1["face_index_map"]), "face_index_map"
    assert torch.equal(m0["weight_map"], m1["weight_map"]), "weight_map"
    assert torch.equal(i0, i1), "images"
    for k in L0:
        check_same(L1[k].grad, L0[k].grad, det, "grad " + k)


@pytest.mark.parametrize("mode", ["tiles", "fine", "dense", "unstaged", "deterministic"])
@pytest.mark.parametrize("name", lg.FIXTURES)
def test_same_topology_lit_with_light_gradients(nr, unstaged, name, mode):
    """Lights with light gradients and a background picture: per-view faces equal shared faces."""
    d = lg._load(name)
    det = mode == "deterministic"
    unstaged(mode == "unstaged")
    dev = "cuda:0"
    S, aa = int(d["image_size"]), bool(d["anti_aliasing"])
    B = d["vertices"].shape[0]
    R = 2 * S if aa else S
    bg = torch.rand((B, 3, R, R), generator=torch.Generator().manual_seed(3)).to(dev)
    G = torch.from_numpy(d["grad_images"]).to(dev)
    hooks = dict(fine=dict(FORCE_FINE_TILES=True), dense=dict(FORCE_DENSE_RASTER=True)).get(mode, {})
    out = []
    for view_faces in (False, True):
        L = leaves(d, dev, ["vertices", "vertices_textures", "textures"])
        P = lg._light_params(d, dev, True)
        f, ft = torch.from_numpy(d["faces"]).to(dev), torch.from_numpy(d["faces_textures"]).to(dev)
        if view_faces:
            f, ft = per_view(f, B), per_view(ft, B)
        bgl = bg.clone().requires_grad_(True)
        with _Hooks(**hooks):
            images, maps = render(nr, "rgb", S, aa, L["vertices"], f, L["vertices_textures"], ft, L["textures"], G,
                                  lights=lg._lights(nr, P, bool(d["light_backside"])), det=det,
                                  backside=bool(d["draw_backside"]), backgrounds=bgl)
        out.append((images, maps, L, P, bgl))
    (i0, m0, L0, P0, b0), (i1, m1, L1, P1, b1) = out
    assert torch.equal(m0["face_index_map"], m1["face_index_map"])
    if det:
        assert torch.equal(i0, i1), "lit images"
    else:       # the vertex normals are summed with float atomics (index_add)
        np.testing.assert_allclose(i1.cpu().numpy(), i0.cpu().numpy(), rtol=1e-5, atol=1e-6)
    for k in L0:
        check_same(L1[k].grad, L0[k].grad, det, "grad " + k)
    for k in lg.LIGHT_KEYS:
        check_same(P1[k].grad, P0[k].grad, det, "grad light " + k)
    assert torch.equal(b0.grad, b1.grad)


# ---------------------------------------------------------------------------------------------------------------- 2
TEX_H, TEX_W = 12, 8       # the textured model's texture (tests/golden/textured)


def meshes(nr):
    """[(name, vertices [nv,3] world or screen space, faces [nf,3], vt [nvt,2], ft [nf,3], texture [3,H,W], screen)]"""
    g = torch.Generator().manual_seed(11)
    out = []
    d = np.load(os.path.join(GOLDEN, "teapot.npz"))
    for name, v, f in (("teapot", torch.from_numpy(d["vertices"]), torch.from_numpy(d["faces"])),
                       ("sphere",) + bench.sphere_mesh(12)):
        vt = torch.rand((v.shape[0], 2), generator=g) * torch.tensor([TEX_W - 1., TEX_H - 1.])
        out.append((name, v.float(), f.int(), vt, f.int(), torch.rand((3, TEX_H, TEX_W), generator=g), False))
    v, f, vt, ft, tex = nr.load_obj(os.path.join(GOLDEN, "textured", "m.obj"), load_textures=True)
    assert tex.shape == (3, TEX_H, TEX_W)
    out.append(("textured", torch.from_numpy(v), torch.from_numpy(f).int(), torch.from_numpy(vt),
                torch.from_numpy(ft).int(), torch.from_numpy(np.ascontiguousarray(tex)).float(), False))
    tri = torch.from_numpy(random_triangles(1, 500, 5, size=0.08)[0])          # [nf,3,3] screen space
    nf = tri.shape[0]
    vt = torch.rand((3 * nf, 2), generator=g) * torch.tensor([TEX_W - 1., TEX_H - 1.])
    idx = torch.arange(3 * nf, dtype=torch.int32).reshape(nf, 3)
    out.append(("random", tri.reshape(-1, 3), idx, vt, idx, torch.rand((3, TEX_H, TEX_W), generator=g), True))
    return out


def screen_views(nr, ms, k):
    """k rounds of the meshes, every view with its own camera -> list of (mesh index, screen vertices [nv,3])"""
    g = torch.Generator().manual_seed(k)
    views = []
    for r in range(k):
        for i, m in enumerate(ms):
            v = m[1]
            if not m[6]:
                eye = nr.get_points_from_angles(torch.full((1,), 2.732), torch.rand(1, generator=g) * 60 - 20,
                                                torch.rand(1, generator=g) * 360)
                v = nr.perspective(nr.look_at(v[None], eye))[0]
            views.append((i, v.contiguous()))
    return views


def pad_batch(ms, views):
    """Padded per-view batch: vertices / vt padded with junk, faces / ft with [0, 0, 0]."""
    nv = max(v.shape[0] for _, v in views)
    nf = max(ms[i][2].shape[0] for i, _ in views)
    nvt = max(ms[i][3].shape[0] for i, _ in views)
    B = len(views)
    V = torch.full((B, nv, 3), 0.25)
    F = torch.zeros((B, nf, 3), dtype=torch.int32)
    VT = torch.full((B, nvt, 2), 1.5)
    FT = torch.zeros((B, nf, 3), dtype=torch.int32)
    T = torch.empty((B, 3, TEX_H, TEX_W))
    for b, (i, v) in enumerate(views):
        _, _, f, vt, ft, tex, _ = ms[i]
        V[b, :v.shape[0]] = v
        F[b, :f.shape[0]] = f
        VT[b, :vt.shape[0]] = vt
        FT[b, :ft.shape[0]] = ft
        T[b] = tex
    return V, F, VT, FT, T


@pytest.mark.parametrize("path", ["binview", "general", "8x8", "dense", "deterministic"])
@pytest.mark.parametrize("mode", ["rgba", "silhouettes", "depth", "lit"])
def test_distinct_meshes_equal_single_view_calls(nr, mode, path):
    dev = "cuda:0"
    S = 64
    ms = meshes(nr)
    views = screen_views(nr, ms, 1)
    if path == "8x8":
        # enough rounds of the four meshes that k_raster runs 8x8 blocks on the batch
        fims = []
        for i, v in views:
            f = ms[i][2].long()
            fims.append(oracle.face_index_map(v[f][None].numpy(), S, 0.1, 100.0, True)[0])
        k = copies(np.stack(fims), "8x8", fine=False)
        views = screen_views(nr, ms, k)
    det = path == "deterministic"
    lit = mode == "lit"
    rmode = "rgb" if lit else mode
    rgb = rmode in ("rgb", "rgba")
    V, F, VT, FT, T = pad_batch(ms, views)
    B = V.shape[0]
    G = torch.randn((B, 5, S, S), generator=torch.Generator().manual_seed(2)).to(dev)
    C = {"rgba": 4, "rgb": 3}.get(rmode, 1)
    G = G[:, :C]

    def lights(sel):
        g = torch.Generator().manual_seed(9)
        col = torch.rand((B, 3), generator=g).to(dev)[sel]
        dirn = (torch.tensor([0., 0., -1.]) + 0.3 * torch.randn((B, 3), generator=g)).to(dev)[sel]
        return [nr.DirectionalLight(col, dirn), nr.AmbientLight(0.5 * col)]

    hooks = dict(PATHS.get(path, {}))
    Vb = V.to(dev).requires_grad_(True)
    VTb = VT.to(dev).requires_grad_(True)
    Tb = T.to(dev).requires_grad_(True)
    with _Hooks(**hooks):
        ib, mb = render(nr, rmode, S, False, Vb, F.to(dev), VTb if rgb else None, FT.to(dev) if rgb else None,
                        Tb if rgb else None, G, lights=lights(slice(None)) if lit else None, det=det)
    fim_b = mb["face_index_map"].cpu().numpy()
    for b, (i, v) in enumerate(views):
        _, _, f, vt, ft, tex, _ = ms[i]
        nv, nf, nvt = v.shape[0], f.shape[0], vt.shape[0]
        v1 = v[None].to(dev).requires_grad_(True)
        vt1 = vt[None].to(dev).requires_grad_(True)
        t1 = tex[None].to(dev).requires_grad_(True)
        with _Hooks(**hooks):
            i1, m1 = render(nr, rmode, S, False, v1, f.to(dev), vt1 if rgb else None, ft.to(dev) if rgb else None,
                            t1 if rgb else None, G[b:b + 1], lights=lights(slice(b, b + 1)) if lit else None, det=det)
        assert np.array_equal(fim_b[b], m1["face_index_map"][0].cpu().numpy()), "view %d: face_index_map" % b
        assert fim_b[b].max() < nf, "view %d: a padded face was drawn" % b
        # the C oracle on the view's own gathered faces
        want = oracle.face_index_map(v[f.long()][None].numpy(), S, 0.1, 100.0, True)[0]
        assert np.array_equal(fim_b[b], want), "view %d: face_index_map vs the oracle" % b
        if lit:
            np.testing.assert_allclose(ib[b].cpu().numpy(), i1[0].cpu().numpy(), rtol=1e-5, atol=1e-6)
        else:
            assert torch.equal(ib[b], i1[0]), "view %d: images" % b
        exact = det and not lit
        check_same(Vb.grad[b, :nv], v1.grad[0], exact, "view %d grad_vertices" % b)
        assert not Vb.grad[b, nv:].any(), "view %d: padded vertices got a gradient" % b
        if rgb:
            check_same(Tb.grad[b], t1.grad[0], exact, "view %d grad_textures" % b)
            check_same(VTb.grad[b, :nvt], vt1.grad[0], exact, "view %d grad_vertices_textures" % b)
            assert not VTb.grad[b, nvt:].any(), "view %d: padded texture vertices got a gradient" % b


def test_distinct_meshes_dense_path(nr):
    """A dense batch (z-buffer path) of different random meshes, each view against its own single-view call and the
    oracle; the path is asserted from the call's statistics."""
    from neural_renderer_v2_pytorch_b200 import rasterize as rz
    dev, S = "cuda:0", 128
    tris = [random_triangles(1, n, 40 + n, size=0.02)[0] for n in (6000, 4000, 5000)]
    nf = max(t.shape[0] for t in tris)
    B = len(tris)
    V = torch.full((B, 3 * nf, 3), -0.5)
    F = torch.zeros((B, nf, 3), dtype=torch.int32)
    for b, t in enumerate(tris):
        V[b, :3 * t.shape[0]] = torch.from_numpy(t).reshape(-1, 3)
        F[b, :t.shape[0]] = torch.arange(3 * t.shape[0], dtype=torch.int32).reshape(-1, 3)
    G = torch.randn((B, 1, S, S), generator=torch.Generator().manual_seed(1)).to(dev)
    Vb = V.to(dev).requires_grad_(True)
    with _Hooks(FORCE_DENSE_RASTER=True):
        ib, mb = render(nr, "silhouettes", S, False, Vb, F.to(dev), G=G)
        sc = rz._Scratch.get(torch.device(dev), torch.cuda.current_stream().cuda_stream)
        assert sc.last_dense, "the call did not take the z-buffer path"
        for b, t in enumerate(tris):
            n = t.shape[0]
            v1 = torch.from_numpy(t).reshape(1, -1, 3).to(dev).requires_grad_(True)
            f1 = torch.arange(3 * n, dtype=torch.int32, device=dev).reshape(-1, 3)
            i1, m1 = render(nr, "silhouettes", S, False, v1, f1, G=G[b:b + 1])
            assert torch.equal(mb["face_index_map"][b], m1["face_index_map"][0])
            assert np.array_equal(mb["face_index_map"][b].cpu().numpy(), oracle.face_index_map(t[None], S, 0.1, 100.0, True)[0])
            assert torch.equal(ib[b], i1[0])
            grad_close(Vb.grad[b, :3 * n].cpu().numpy(), v1.grad[0].cpu().numpy(), "grad_vertices")
            assert not Vb.grad[b, 3 * n:].any()


def test_textured_view_matches_the_oracle_pipeline(nr):
    """The textured teapot inside a padded batch of distinct meshes: its view against oracle.pipeline on images and
    gradients.  (The textured model's UVs reach outside its texture: the oracle raises IndexError there, as the
    reference does, while the kernels read zeros.)"""
    dev, S = "cuda:0", 64
    ms = meshes(nr)
    views = screen_views(nr, ms, 1)
    V, F, VT, FT, T = pad_batch(ms, views)
    B = V.shape[0]
    b = [n for n, *_ in ms].index("teapot")
    i, v = views[b]
    _, _, f, vt, ft, tex, _ = ms[i]
    G = torch.randn((B, 4, S, S), generator=torch.Generator().manual_seed(5))
    Vb, Tb = V.to(dev).requires_grad_(True), T.to(dev).requires_grad_(True)
    ib, _ = render(nr, "rgba", S, False, Vb, F.to(dev), VT.to(dev), FT.to(dev), Tb, G.to(dev))
    v0, t0 = v[None].clone().requires_grad_(True), tex[None].clone().requires_grad_(True)
    img0 = ref.rasterize(v0, f.numpy(), S, False, draw_rgb=True, draw_silhouettes=True, vertices_textures=vt[None],
                         faces_textures=ft.numpy(), textures=t0)
    (img0 * G[b:b + 1]).sum().backward()
    np.testing.assert_allclose(ib[b].cpu().numpy(), img0[0].detach().numpy(), rtol=1e-5, atol=1e-6)
    grad_close(Vb.grad[b, :v.shape[0]].cpu().numpy(), v0.grad[0].numpy(), "grad_vertices")
    grad_close(Tb.grad[b].cpu().numpy(), t0.grad[0].numpy(), "grad_textures")


# ---------------------------------------------------------------------------------------------------------------- 4
@pytest.mark.parametrize("which", ["faces", "faces_textures"])
def test_mixed_forms_equal_fully_per_view(nr, which):
    dev, S, B = "cuda:0", 64, 3
    d = np.load(os.path.join(GOLDEN, "teapot.npz"))
    g = torch.Generator().manual_seed(4)
    f = torch.from_numpy(d["faces"]).int()
    eye = nr.get_points_from_angles(torch.full((B,), 2.732), torch.rand(B, generator=g) * 60, torch.rand(B, generator=g) * 360)
    v = nr.perspective(nr.look_at(torch.from_numpy(d["vertices"])[None].repeat(B, 1, 1), eye)).to(dev)
    vt_np, ft_np, tex_np = nr.create_textures(f.shape[0], 2)
    tex = torch.rand((B,) + tex_np.shape, generator=g).to(dev)
    vt = torch.from_numpy(vt_np)[None].repeat(B, 1, 1).to(dev)
    ft = torch.from_numpy(ft_np).int().to(dev)
    # per-view rows that really differ: every view pads a different third of the faces / retargets a third of the
    # texture faces
    F, FT = per_view(f, B).clone(), per_view(ft.cpu(), B).clone()
    for b in range(B):
        F[b, b::3] = 0
        FT[b, b::3] = FT[b, 0]
    F, FT, f = F.to(dev), FT.to(dev), f.to(dev)
    G = torch.randn((B, 4, S, S), generator=g).to(dev)
    if which == "faces":        # per-view faces, shared faces_textures
        mixed, full = (F, ft), (F, per_view(ft, B))
    else:                       # shared faces, per-view faces_textures
        mixed, full = (f, FT), (per_view(f, B), FT)
    out = []
    for ff, fft in (full, mixed):
        v1, t1 = v.clone().requires_grad_(True), tex.clone().requires_grad_(True)
        images, maps = render(nr, "rgba", S, False, v1, ff, vt, fft, t1, G, det=True)
        out.append((images, maps, v1.grad, t1.grad))
    (i0, m0, gv0, gt0), (i1, m1, gv1, gt1) = out
    assert torch.equal(m0["face_index_map"], m1["face_index_map"])
    assert torch.equal(i0, i1)
    assert torch.equal(gv0, gv1) and torch.equal(gt0, gt1)


# ---------------------------------------------------------------------------------------------------------------- 5
def test_out_of_range_index_in_one_view_raises(nr):
    dev = "cuda:0"
    hp = nr.RasterizeHyperparam(image_size=32, anti_aliasing=False)
    v = torch.rand((3, 4, 3), device=dev)
    f = torch.tensor([[0, 1, 2], [1, 2, 3]], dtype=torch.int32)[None].repeat(3, 1, 1)
    f[2, 1, 2] = 4
    with pytest.raises(IndexError):
        nr.rasterize_silhouettes(v, f.to(dev), nr.RasterizeParam(), hp)
    ft = torch.tensor([[0, 1, 2], [1, 2, 3]], dtype=torch.int32)[None].repeat(3, 1, 1)
    ft[1, 0, 0] = -1
    p = nr.RasterizeParam(vertices_textures=torch.rand((3, 4, 2), device=dev), faces_textures=ft.to(dev),
                          textures=torch.rand((3, 3, 4, 4), device=dev))
    with pytest.raises(IndexError):
        nr.rasterize_rgb(v, f.clamp(max=3).to(dev), p, hp)


def test_view_faces_flag_without_faces_is_rejected(nr):
    from neural_renderer_v2_pytorch_b200 import _lib
    L = _lib.lib()
    cfg = _lib.RasterConfig(batch=1, num_vertices=3, num_faces=1, image_size=16,
                            flags=_lib.NR_DRAW_SILHOUETTES | _lib.NR_VIEW_FACES, near_plane=0.1, far_plane=100., eps=1e-5,
                            depth_min_delta=1e-4)
    v = torch.rand((1, 3, 3), device="cuda")
    fim = torch.empty((1, 16, 16), dtype=torch.int32, device="cuda")
    img = torch.empty((1, 1, 16, 16), device="cuda")
    tl = torch.empty(8 + 16, dtype=torch.int32, device="cuda")
    ws = torch.empty(int(L.nr_workspace_bytes(ctypes.byref(cfg), 1024)) + 256, dtype=torch.uint8, device="cuda")
    base = (ws.data_ptr() + 255) & ~255
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = L.nr_rasterize_forward(ctypes.byref(cfg), p(v), None, None, None, None, p(fim), None, None, p(img), None, None,
                                p(tl), ctypes.c_void_p(base), ws.numel() - (base - ws.data_ptr()), 1024, None, None, None,
                                None, s)
    assert rc == _lib.NR_ERR_INVALID_ARGUMENT
    gv = torch.zeros_like(v)
    rc = L.nr_rasterize_backward_lights(ctypes.byref(cfg), p(v), None, None, None, None, p(fim), p(img), None, None,
                                        p(img), p(gv), None, None, None, None, None, None, s)
    assert rc == _lib.NR_ERR_INVALID_ARGUMENT
    rc = L.nr_rasterize_backward(ctypes.byref(cfg), p(v), None, None, None, None, p(fim), p(img), None, None,
                                 p(img), p(gv), None, None, None, None, s)
    assert rc == _lib.NR_ERR_INVALID_ARGUMENT


# ---------------------------------------------------------------------------------------------------------------- 6
def test_mesh_get_batch_renders(nr):
    dev, B, S = "cuda:0", 4, 64
    mesh = nr.Mesh(os.path.join(GOLDEN, "textured", "m.obj")).to(dev)
    v, f, _ = mesh.get_batch(B)
    assert f.shape == (B, mesh.num_faces, 3)
    eye = nr.get_points_from_angles(torch.full((B,), 2.732), torch.linspace(-20, 40, B), torch.linspace(0, 300, B)).to(dev)
    vs = nr.perspective(nr.look_at(v, eye))
    hp = lambda: nr.RasterizeHyperparam(image_size=S, anti_aliasing=True)
    a = nr.rasterize_silhouettes(vs, f, nr.RasterizeParam(), hp())
    b = nr.rasterize_silhouettes(vs, mesh.faces, nr.RasterizeParam(), hp())
    assert a.shape == (B, S, S) and a.sum() > 0
    assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------- 7
def test_shared_mesh_with_per_view_face_subsets(nr):
    """One [1, nv, 3] mesh through Renderer.render_silhouettes (fused camera) with [B, 3] viewpoints and a different
    face subset per view: its gradient is the sum of the single-view calls."""
    dev, B, S = "cuda:0", 4, 64
    d = np.load(os.path.join(GOLDEN, "teapot.npz"))
    g = torch.Generator().manual_seed(8)
    f = torch.from_numpy(d["faces"]).int()
    F = per_view(f, B).clone()
    for b in range(B):
        F[b, torch.rand(f.shape[0], generator=g) < 0.3] = 0
    eye = nr.get_points_from_angles(torch.full((B,), 2.732), torch.rand(B, generator=g) * 60, torch.rand(B, generator=g) * 360)
    G = torch.randn((B, S, S), generator=g).to(dev)
    r = nr.Renderer()
    r.image_size, r.anti_aliasing = S, False
    r.viewpoints = eye.to(dev)
    mesh = torch.from_numpy(d["vertices"])[None].to(dev).requires_grad_(True)
    img = r.render_silhouettes(mesh, F.to(dev))
    (img * G).sum().backward()
    total = torch.zeros_like(mesh)
    for b in range(B):
        r.viewpoints = eye[b:b + 1].to(dev)
        m1 = torch.from_numpy(d["vertices"])[None].to(dev).requires_grad_(True)
        i1 = r.render_silhouettes(m1, F[b].to(dev))
        (i1 * G[b:b + 1]).sum().backward()
        assert torch.equal(img[b], i1[0]), "view %d" % b
        total += m1.grad
    grad_close(mesh.grad.cpu().numpy(), total.cpu().numpy(), "shared mesh gradient")


# ---------------------------------------------------------------------------------------------------------------- 8
def test_capture_step_with_per_view_faces(nr):
    dev, S = "cuda:0", 64
    ms = meshes(nr)
    V, F, VT, FT, T = pad_batch(ms, screen_views(nr, ms, 2))
    B = V.shape[0]
    v = V.to(dev).requires_grad_(True)
    tex = T.to(dev).requires_grad_(True)
    vt, F, FT = VT.to(dev), F.to(dev), FT.to(dev)
    G = torch.randn((B, 4, S, S), generator=torch.Generator().manual_seed(6)).to(dev)

    def step():
        hp = nr.RasterizeHyperparam(image_size=S, anti_aliasing=False)
        hp.deterministic = True
        img = nr.rasterize_rgba(v, F, nr.RasterizeParam(vertices_textures=vt, faces_textures=FT, textures=tex), hp)
        (img * G).sum().backward()
        return img

    replay = nr.capture_step(step, params=[v, tex], warmup=2)
    img = replay().detach().clone()
    torch.cuda.synchronize()
    gv, gt = v.grad.clone(), tex.grad.clone()
    v.grad = tex.grad = None
    eager = step().detach()
    assert torch.equal(img, eager)
    assert torch.equal(gv, v.grad) and torch.equal(gt, tex.grad)


# ---------------------------------------------------------------------------------------------------------------- 9
@pytest.mark.parametrize("path", ["binview", "general", "fine", "dense", "8x8"])
def test_kernels_stay_inside_their_buffers_with_per_view_faces(nr, path):
    """Every output of forward and backward carved out of a poisoned allocation, per-view faces: the guard words
    on both sides survive, and the result equals the public API's."""
    from neural_renderer_v2_pytorch_b200 import _lib
    L = _lib.lib()
    dev, S, G_ = "cuda:0", 64, 4096
    ms = meshes(nr)
    views = screen_views(nr, ms, 1)
    fine, dense = path == "fine", path == "dense"
    if path == "8x8":
        fims = [oracle.face_index_map(v[ms[i][2].long()][None].numpy(), S, 0.1, 100.0, True)[0] for i, v in views]
        views = screen_views(nr, ms, copies(np.stack(fims), "8x8", fine=False))
    V, F, VT, FT, T = (t.to(dev).contiguous() for t in pad_batch(ms, views))
    B, nv, nf = V.shape[0], V.shape[1], F.shape[1]
    flags = (_lib.NR_DRAW_RGB | _lib.NR_DRAW_SILHOUETTES | _lib.NR_DRAW_BACKSIDE | _lib.NR_VIEW_FACES |
             (_lib.NR_FINE_TILES if fine else 0) | (_lib.NR_GENERAL_BINNING if path in ("general", "fine", "dense") else 0) |
             (_lib.NR_DENSE_RASTER if dense else 0))
    cfg = _lib.RasterConfig(batch=B, num_vertices=nv, num_faces=nf, image_size=S, flags=flags, near_plane=0.1,
                            far_plane=100., eps=1e-5, depth_min_delta=1e-4, num_tex_vertices=VT.shape[1],
                            tex_height=TEX_H, tex_width=TEX_W)
    tile = 8 if fine else 16
    ntx = (S + tile - 1) // tile
    cap = 8 * B * nf
    PI, PF = 0x5a5a5a5a, 12345.5

    def guarded(n, dtype):
        big = torch.full((n + 2 * G_,), PI if dtype == torch.int32 else PF, dtype=dtype, device=dev)
        return big, big[G_:G_ + n]

    sizes = dict(fim=(B * S * S, torch.int32), images=(B * 4 * S * S, torch.float32),
                 tile_list=(8 + 16 * B * ntx * ntx, torch.int32), gv=(V.numel(), torch.float32),
                 gtex=(T.numel(), torch.float32), gvt=(VT.numel(), torch.float32),
                 ws=(int(L.nr_workspace_bytes(ctypes.byref(cfg), cap)) // 4 + 64, torch.int32))
    buf = {k: guarded(n, dt) for k, (n, dt) in sizes.items()}
    for k in ("gv", "gtex", "gvt"):
        buf[k][1].zero_()
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    ws = buf["ws"][1]
    base = (ws.data_ptr() + 255) & ~255
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = L.nr_rasterize_forward(ctypes.byref(cfg), p(V), p(F), p(VT), p(FT), p(T), p(buf["fim"][1]), None, None,
                                p(buf["images"][1]), None, None, p(buf["tile_list"][1]), ctypes.c_void_p(base),
                                ws.numel() * 4 - (base - ws.data_ptr()), cap, None, None, None, None, s)
    _lib.check(rc, "forward")
    Gr = torch.randn((B, 4, S, S), generator=torch.Generator().manual_seed(1)).to(dev)
    rc = L.nr_rasterize_backward(ctypes.byref(cfg), p(V), p(F), p(VT), p(FT), p(T), p(buf["fim"][1]), p(buf["images"][1]),
                                 None, None if fine else p(buf["tile_list"][1]), p(Gr), p(buf["gv"][1]), p(buf["gtex"][1]),
                                 p(buf["gvt"][1]), None, None, s)
    _lib.check(rc, "backward")
    torch.cuda.synchronize()
    for k, (n, _) in sizes.items():
        big = buf[k][0]
        want = PI if big.dtype == torch.int32 else PF
        assert bool((big[:G_] == want).all()) and bool((big[G_ + n:] == want).all()), "%s: guard words overwritten" % k
    assert not (buf["fim"][1] == PI).any() and not (buf["images"][1] == PF).any()
    assert float(buf["gv"][1].abs().sum()) > 0 and float(buf["gtex"][1].abs().sum()) > 0
    hp = nr.RasterizeHyperparam(image_size=S, anti_aliasing=False)
    img = nr.rasterize_rgba(V, F, nr.RasterizeParam(vertices_textures=VT, faces_textures=FT, textures=T), hp)
    assert torch.equal(img.reshape(-1), buf["images"][1])
