"""Per-face texture cubes: textures [B, nf, ts, ts, ts, 3] with no uv inputs (NR_FACE_TEXTURES, the texture format of
Mesh.get_batch) through both binning paths, 8x8 tiles, the z-buffer path, both k_raster block heights, the staged,
unstaged and deterministic backward, lights, backgrounds and per-view faces.

The definition is face_textures_oracle (the oracle pipeline with the trilinear per-face sample); bars as elsewhere in
the suite: face_index_map bit for bit, images rtol 1e-5 / atol 1e-6, gradients |d| <= 1e-5 |ref| + 1e-5 max |ref|."""
import ctypes
import os

import numpy as np
import pytest
import torch

import oracle
from face_textures_oracle import rasterize as fref
from test_gpu_parity import CASES, GOLDEN, grad_close, random_triangles
from test_gpu_raster_blocks import _Hooks, copies
import test_gpu_light_gradients as lg

pytestmark = pytest.mark.gpu

UNSTAGED = "NR_FORCE_UNSTAGED_BACKWARD"
HOOKS = {"general": dict(FORCE_GENERAL_BINNING=True), "fine": dict(FORCE_FINE_TILES=True),
         "dense": dict(FORCE_DENSE_RASTER=True)}
PATHS = ["binview", "general", "fine", "dense", "8x8", "unstaged", "deterministic"]


@pytest.fixture(scope="module")
def nr():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import neural_renderer_v2_pytorch_b200 as nr_
    return nr_


def load(name, ts, seed=0):
    """Geometry of a golden case, random cubes [B, nf, ts, ts, ts, 3], random upstream gradient [B, 4, S, S]."""
    d = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    B, nf, S = d["vertices"].shape[0], d["faces"].shape[0], int(d["image_size"])
    g = torch.Generator().manual_seed(1000 * ts + seed)
    tex = torch.rand((B, nf, ts, ts, ts, 3), generator=g)
    G = torch.randn((B, 4, S, S), generator=g)
    return d, tex, G


def hyper(nr, d, mode=None, det=False):
    hp = nr.RasterizeHyperparam(image_size=int(d["image_size"]), near=float(d["near"]), far=float(d["far"]),
                                anti_aliasing=bool(d["anti_aliasing"]), draw_backside=bool(d["draw_backside"]))
    if mode is not None:
        hp.draw_rgb, hp.draw_silhouettes, hp.draw_depth = True, mode == "rgba", False
    hp.deterministic = det
    return hp


def channels(mode, G):
    return G if mode == "rgba" else G[:, :3]


def gpu_run(nr, d, tex, mode, G, det=False, lights=None, backgrounds=None, verts=None, faces=None):
    """The public API on cuda:0 -> (images, grad vertices, grad textures, face_index_map), all on the CPU; lights /
    backgrounds as given (their gradients land in their own leaves)."""
    dev = "cuda:0"
    v = (torch.from_numpy(d["vertices"]) if verts is None else verts).to(dev).requires_grad_(True)
    f = torch.from_numpy(d["faces"]).to(dev) if faces is None else faces.to(dev)
    t = tex.to(dev).requires_grad_(True)
    p = nr.RasterizeParam(textures=t, lights=lights, backgrounds=backgrounds)
    images = (nr.rasterize_rgba if mode == "rgba" else nr.rasterize_rgb)(v, f, p, hyper(nr, d, det=det))
    (images * channels(mode, G).to(dev)).sum().backward()
    maps = nr.rasterize_maps(v.detach(), f, p, hyper(nr, d, mode, det))
    torch.cuda.synchronize()
    return images.detach().cpu(), v.grad.cpu(), t.grad.cpu(), maps["face_index_map"].cpu()


def oracle_run(d, tex, mode, G, lights=None, backgrounds=None):
    v = torch.from_numpy(d["vertices"]).requires_grad_(True)
    t = tex.clone().requires_grad_(True)
    img, maps = fref(v, d["faces"], int(d["image_size"]), bool(d["anti_aliasing"]), t, near=float(d["near"]),
                     far=float(d["far"]), draw_backside=bool(d["draw_backside"]), draw_silhouettes=mode == "rgba",
                     lights=lights, backgrounds=backgrounds, return_maps=True)
    (img * channels(mode, G)).sum().backward()
    return img.detach(), v.grad, t.grad, maps["face_index_map"]


def check(got, want, k=1):
    """got = gpu_run of k copies of the views of want = oracle_run."""
    rep = lambda x: np.concatenate([np.asarray(x)] * k)
    img, gv, gt, fim = got
    wimg, wgv, wgt, wfim = want
    assert np.array_equal(fim.numpy(), rep(wfim)), "face_index_map not bit-exact"
    np.testing.assert_allclose(img.numpy(), rep(wimg), rtol=1e-5, atol=1e-6)
    grad_close(gv.numpy(), rep(wgv), "grad_vertices")
    grad_close(gt.numpy(), rep(wgt), "grad_textures")
    assert np.abs(rep(wgt)).max() > 0


def run_path(nr, path, d, tex, mode, G, monkeypatch):
    """gpu_run on one raster / backward path -> (result, copies)."""
    k = 1
    if path == "8x8":
        R = int(d["image_size"]) * (2 if bool(d["anti_aliasing"]) else 1)
        f = np.ascontiguousarray(d["vertices"][:, d["faces"]], dtype=np.float32)
        k = copies(oracle.face_index_map(f, R, float(d["near"]), float(d["far"]), bool(d["draw_backside"])), "8x8", False)
        d = dict(d, vertices=np.concatenate([d["vertices"]] * k))
        tex, G = torch.cat([tex] * k), torch.cat([G] * k)
    if path == "unstaged":
        monkeypatch.setenv(UNSTAGED, "1")
    with _Hooks(**HOOKS.get(path, {})):
        out = gpu_run(nr, d, tex, mode, G, det=path == "deterministic")
    return out, k


# ---------------------------------------------------------------------------------------------------------------- 1
@pytest.mark.parametrize("mode", ["rgb", "rgba"])
@pytest.mark.parametrize("name", CASES)
def test_golden_geometry(nr, name, mode):
    """Every golden case's geometry (anti-aliased or not, culled, clipped) with random cubes vs the oracle."""
    d, tex, G = load(name, 4)
    check(gpu_run(nr, d, tex, mode, G), oracle_run(d, tex, mode, G))


@pytest.mark.parametrize("ts", [1, 2, 4, 7])
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name,mode", [("case_rgba_64", "rgba"), ("case_rgba_aa_32", "rgb")])
def test_every_path(nr, name, mode, path, ts, monkeypatch):
    d, tex, G = load(name, ts, seed=1)
    got, k = run_path(nr, path, d, tex, mode, G, monkeypatch)
    if path == "8x8":
        assert k > 1
    check(got, oracle_run(d, tex, mode, G), k)


def test_deterministic_runs_are_bit_identical(nr):
    d, tex, G = load("case_rgba_64", 4, seed=2)
    a = gpu_run(nr, d, tex, "rgba", G, det=True)
    b = gpu_run(nr, d, tex, "rgba", G, det=True)
    for x, y, what in zip(a, b, ("images", "grad_vertices", "grad_textures", "face_index_map")):
        assert torch.equal(x, y), what


# ---------------------------------------------------------------------------------------------------------------- 2
@pytest.mark.parametrize("det", [False, True])
@pytest.mark.parametrize("name", lg.FIXTURES)
def test_lights_with_light_gradients(nr, name, det):
    """Directional, ambient and specular lights multiply the cube sample; gradients reach the light parameters."""
    d = dict(lg._load(name))
    B, nf = d["vertices"].shape[0], d["faces"].shape[0]
    g = torch.Generator().manual_seed(3)
    tex = torch.rand((B, nf, 3, 3, 3, 3), generator=g)
    G = torch.randn((B, 4, int(d["image_size"]), int(d["image_size"])), generator=g)
    lb = bool(d["light_backside"])
    P = lg._light_params(d, "cuda:0", True)
    with lg._Mode("tiles"):
        img, gv, gt, fim = gpu_run(nr, d, tex, "rgb", G, det=det, lights=lg._lights(nr, P, lb))
    Q = lg._light_params(d, "cpu", True)
    wimg, wgv, wgt, wfim = oracle_run(d, tex, "rgb", G, lights=lg._oracle_lights(Q, lb))
    assert np.array_equal(fim.numpy(), wfim.numpy())
    np.testing.assert_allclose(img.numpy(), wimg.numpy(), rtol=1e-5, atol=2e-6)
    grad_close(gt.numpy(), wgt.numpy(), "grad_textures")
    # the normal path goes through torch index_add and powf: 1e-4 of the scale (test_gpu_parity.test_lights_golden)
    assert np.abs(gv.numpy() - wgv.numpy()).max() <= 1e-4 * np.abs(wgv.numpy()).max()
    for k in lg.LIGHT_KEYS:
        want = Q[k].grad.numpy()
        got = P[k].grad.cpu().numpy()
        assert np.abs(got - want).max() <= 1e-4 * max(np.abs(want).max(), 1e-12), k


@pytest.mark.parametrize("name", ["case_rgba_64", "case_rgba_aa_32"])
def test_backgrounds(nr, name):
    d, tex, G = load(name, 2, seed=4)
    B, S = d["vertices"].shape[0], int(d["image_size"])
    R = S * (2 if bool(d["anti_aliasing"]) else 1)
    bg = torch.rand((B, 3, R, R), generator=torch.Generator().manual_seed(5))
    bg_gpu = bg.cuda().requires_grad_(True)
    got = gpu_run(nr, d, tex, "rgba", G, backgrounds=bg_gpu)
    bg_cpu = bg.clone().requires_grad_(True)
    check(got, oracle_run(d, tex, "rgba", G, backgrounds=bg_cpu))
    grad_close(bg_gpu.grad.cpu().numpy(), bg_cpu.grad.numpy(), "grad_backgrounds")


# ---------------------------------------------------------------------------------------------------------------- 3
def test_per_view_faces_equal_single_view_calls(nr):
    """Distinct meshes padded to a common nv / nf ([0, 0, 0] faces), [B, nf, 3] faces with their cubes: every view
    equals a single-view call on its own mesh (images bit for bit), padded cubes get no gradient, and the oracle."""
    S, ts, nfs = 64, 3, [40, 25, 60]
    B, NF = len(nfs), max(nfs)
    g = torch.Generator().manual_seed(7)
    V = torch.zeros((B, 3 * NF, 3))
    F = torch.zeros((B, NF, 3), dtype=torch.int32)
    for b, n in enumerate(nfs):
        V[b, :3 * n] = torch.from_numpy(random_triangles(1, n, 10 + b, size=0.3)[0].reshape(-1, 3))
        F[b, :n] = torch.arange(3 * n, dtype=torch.int32).reshape(n, 3)
    T = torch.rand((B, NF, ts, ts, ts, 3), generator=g)
    G = torch.randn((B, 4, S, S), generator=g)
    d = dict(image_size=S, near=0.1, far=100., anti_aliasing=False, draw_backside=True)
    img, gv, gt, fim = gpu_run(nr, d, T, "rgba", G, verts=V, faces=F)
    for b, n in enumerate(nfs):
        db = dict(d, vertices=V[b:b + 1, :3 * n].numpy(), faces=F[b, :n].numpy())
        one = gpu_run(nr, db, T[b:b + 1, :n], "rgba", G[b:b + 1])
        assert torch.equal(img[b:b + 1], one[0]), b
        assert torch.equal(fim[b:b + 1], one[3]), b
        grad_close(gv[b:b + 1, :3 * n].numpy(), one[1].numpy(), "grad_vertices %d" % b)
        grad_close(gt[b:b + 1, :n].numpy(), one[2].numpy(), "grad_textures %d" % b)
        assert not gt[b, n:].any() and not gv[b, 3 * n:].any()
        check(one, oracle_run(db, T[b:b + 1, :n], "rgba", G[b:b + 1]))


# ---------------------------------------------------------------------------------------------------------------- 4
def _teapot_mesh(nr, tmp_path, ts, seed):
    d = np.load(os.path.join(GOLDEN, "teapot.npz"))
    path = tmp_path / "teapot.obj"
    with open(path, "w") as fh:
        fh.writelines("v %.8f %.8f %.8f\n" % tuple(p) for p in d["vertices"])
        fh.writelines("f %d %d %d\n" % tuple(f + 1) for f in d["faces"])
    torch.manual_seed(seed)
    return nr.Mesh(str(path), texture_size=ts).to("cuda")


def _eyes(nr, B):
    return nr.get_points_from_angles(torch.full((B,), 2.732), torch.tensor([15., 30., -10.][:B]),
                                     torch.tensor([40., 220., 130.][:B]))


def test_mesh_get_batch_renders_and_learns(nr, tmp_path):
    """Mesh.get_batch end to end through Renderer.render: the gradient of the learnable textures equals the oracle's,
    and an Adam step with set_lr moves them (and not the vertices)."""
    B, S = 3, 64
    mesh = _teapot_mesh(nr, tmp_path, 4, 0)
    r = nr.Renderer()
    r.image_size, r.anti_aliasing = S, True
    r.viewpoints = _eyes(nr, B).cuda()
    v, f, t = mesh.get_batch(B)
    img = r.render(v, f, None, None, t)
    assert img.shape == (B, 4, S, S)
    G = torch.randn(img.shape, generator=torch.Generator().manual_seed(8)).cuda()
    (img * G).sum().backward()
    got = mesh.textures.grad.cpu()
    # the oracle on the screen-space vertices the renderer rasterized
    vs = r.transform_vertices(v).detach().cpu()
    raw = mesh.textures.detach().cpu().requires_grad_(True)
    want_img = fref(vs, f[0].cpu().numpy(), S, True, torch.sigmoid(raw).expand(B, *raw.shape))
    (want_img * G.cpu()).sum().backward()
    np.testing.assert_allclose(img.detach().cpu().numpy(), want_img.detach().numpy(), rtol=1e-5, atol=1e-6)
    grad_close(got.numpy(), raw.grad.numpy(), "mesh.textures.grad")
    before_t, before_v = mesh.textures.detach().clone(), mesh.vertices.clone()
    mesh.set_lr(0., 1.)
    nr.Adam(mesh.parameters(), alpha=0.01).step()
    assert (mesh.textures.detach() - before_t).abs().max() > 1e-3
    assert torch.equal(mesh.vertices, before_v)


def test_texture_fit_reaches_the_oracle_loss(nr, tmp_path):
    """Fixed geometry, target rendered from another cube set, 40 Adam steps (alpha 0.1) on the raw cubes.  The same loop
    on the CPU oracle goes from 3.1e-3 to 1.93e-5; the bar is twice that."""
    d = np.load(os.path.join(GOLDEN, "teapot.npz"))
    B, S, ts, steps = 2, 32, 2, 40
    g = torch.Generator().manual_seed(5)
    vw = torch.from_numpy(d["vertices"])[None].repeat(B, 1, 1)
    eye = nr.get_points_from_angles(torch.full((B,), 2.732), torch.tensor([15., 30.]), torch.tensor([40., 220.]))
    vs = nr.perspective(nr.look_at(vw, eye)).float().cuda()
    faces = torch.from_numpy(d["faces"]).cuda()
    nf = faces.shape[0]
    raw_t = torch.randn((nf, ts, ts, ts, 3), generator=g)
    raw = torch.randn((nf, ts, ts, ts, 3), generator=g).cuda().requires_grad_(True)
    hp = lambda: nr.RasterizeHyperparam(image_size=S, anti_aliasing=False)

    def render(r):
        return nr.rasterize_rgb(vs, faces, nr.RasterizeParam(textures=torch.sigmoid(r).expand(B, *r.shape)), hp())

    with torch.no_grad():
        target = render(raw_t.cuda())
    raw.lr = 1.0
    opt = nr.Adam([raw], alpha=0.1)
    first = None
    for _ in range(steps):
        opt.zero_grad()
        loss = ((render(raw) - target) ** 2).mean()
        first = float(loss.detach()) if first is None else first
        loss.backward()
        opt.step()
    with torch.no_grad():
        final = float(((render(raw) - target) ** 2).mean())
    assert first > 2e-3
    assert final <= 2 * 1.93e-5, final


def test_capture_step_replay_equals_eager(nr):
    d, tex, G = load("case_rgba_64", 4, seed=9)
    dev = "cuda:0"
    v = torch.from_numpy(d["vertices"]).to(dev).requires_grad_(True)
    t = tex.to(dev).requires_grad_(True)
    f = torch.from_numpy(d["faces"]).to(dev)
    Gd = G.to(dev)

    def step():
        hp = hyper(nr, d, det=True)
        img = nr.rasterize_rgba(v, f, nr.RasterizeParam(textures=t), hp)
        (img * Gd).sum().backward()
        return img

    replay = nr.capture_step(step, params=[v, t], warmup=2)
    img = replay().detach().clone()
    torch.cuda.synchronize()
    gv, gt = v.grad.clone(), t.grad.clone()
    v.grad = t.grad = None
    eager = step().detach()
    assert torch.equal(img, eager)
    assert torch.equal(gv, v.grad) and torch.equal(gt, t.grad)


# ---------------------------------------------------------------------------------------------------------------- 5
def _config(_lib, B, nv, nf, S, flags, ts, nvt=0):
    return _lib.RasterConfig(batch=B, num_vertices=nv, num_faces=nf, image_size=S, flags=flags, near_plane=0.1,
                             far_plane=100., eps=1e-5, depth_min_delta=1e-4, num_tex_vertices=nvt, tex_height=ts,
                             tex_width=ts)


@pytest.mark.parametrize("path", ["binview", "general", "fine", "dense", "8x8", "deterministic"])
def test_kernels_stay_inside_their_buffers(nr, path):
    """The cubes and their gradient carved out of poisoned allocations (as every other output): the guard words on
    both sides survive, every gradient entry is written, and the images equal the public API's."""
    from neural_renderer_v2_pytorch_b200 import _lib
    L = _lib.lib()
    d = np.load(os.path.join(GOLDEN, "teapot.npz"))
    B, S, ts, G_ = 3, 64, 3, 4096
    g = torch.Generator().manual_seed(11)
    vw = torch.from_numpy(d["vertices"])[None].repeat(B, 1, 1)
    v = nr.perspective(nr.look_at(vw, _eyes(nr, B))).float().contiguous()
    faces = torch.from_numpy(d["faces"])
    if path == "8x8":
        k = copies(oracle.face_index_map(v[:, faces.long()].numpy(), S), "8x8", False)
        B, v = B * k, torch.cat([v] * k)
    nf = faces.shape[0]
    tex = torch.rand((B, nf, ts, ts, ts, 3), generator=g)
    v, faces, tex = v.cuda(), faces.cuda(), tex.cuda()
    flags = (_lib.NR_DRAW_RGB | _lib.NR_DRAW_SILHOUETTES | _lib.NR_DRAW_BACKSIDE | _lib.NR_FACE_TEXTURES |
             {"general": _lib.NR_GENERAL_BINNING, "fine": _lib.NR_FINE_TILES | _lib.NR_GENERAL_BINNING,
              "dense": _lib.NR_DENSE_RASTER, "deterministic": _lib.NR_DETERMINISTIC}.get(path, 0))
    cfg = _config(_lib, B, v.shape[1], nf, S, flags, ts)
    fine = path == "fine"
    ntx = (S + (8 if fine else 16) - 1) // (8 if fine else 16)
    cap = 8 * B * nf
    POISON_I, POISON_F = 0x5a5a5a5a, 12345.5

    def guarded(n, dtype, fill=None):
        big = torch.full((n + 2 * G_,), POISON_I if dtype == torch.int32 else POISON_F, dtype=dtype, device="cuda")
        if fill is not None:
            big[G_:G_ + n] = fill.reshape(-1)
        return big, big[G_:G_ + n]

    def intact(big, n):
        want = POISON_I if big.dtype == torch.int32 else POISON_F
        return bool((big[:G_] == want).all()) and bool((big[G_ + n:] == want).all())

    sizes = dict(fim=(B * S * S, torch.int32, None), images=(B * 4 * S * S, torch.float32, None),
                 tile_list=(8 + 16 * B * ntx * ntx, torch.int32, None), tex=(tex.numel(), torch.float32, tex),
                 gv=(v.numel(), torch.float32, None), gtex=(tex.numel(), torch.float32, None),
                 ws=(int(L.nr_workspace_bytes(ctypes.byref(cfg), cap)) // 4 + 64, torch.int32, None))
    buf = {k: guarded(n, dt, fill) for k, (n, dt, fill) in sizes.items()}
    ptr = lambda t: ctypes.c_void_p(t.data_ptr())
    zf = _lib.ZeroFill(count=2)
    for i, k in enumerate(("gv", "gtex")):
        zf.ptr[i] = buf[k][1].data_ptr()
        zf.bytes[i] = buf[k][1].numel() * 4
    ws = buf["ws"][1]
    base = (ws.data_ptr() + 255) & ~255
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = L.nr_rasterize_forward(ctypes.byref(cfg), ptr(v), ptr(faces), None, None, ptr(buf["tex"][1]), ptr(buf["fim"][1]),
                                None, None, ptr(buf["images"][1]), None, None, ptr(buf["tile_list"][1]),
                                ctypes.c_void_p(base), ws.numel() * 4 - (base - ws.data_ptr()), cap, None, None,
                                ctypes.byref(zf), None, stream)
    _lib.check(rc, "forward")
    G = torch.randn((B, 4, S, S), generator=g).cuda()
    scratch = None
    if path == "deterministic":
        scratch = torch.zeros(L.nr_deterministic_scratch_bytes(ctypes.byref(cfg)) // 8 + 1, dtype=torch.int64, device="cuda")
    rc = L.nr_rasterize_backward(ctypes.byref(cfg), ptr(v), ptr(faces), None, None, ptr(buf["tex"][1]), ptr(buf["fim"][1]),
                                 ptr(buf["images"][1]), None, None if fine else ptr(buf["tile_list"][1]), ptr(G),
                                 ptr(buf["gv"][1]), ptr(buf["gtex"][1]), None,
                                 ptr(scratch) if scratch is not None else None, None, stream)
    _lib.check(rc, "backward")
    torch.cuda.synchronize()
    for k, (n, _, _) in sizes.items():
        assert intact(buf[k][0], n), "%s: guard words overwritten" % k
    assert not (buf["fim"][1] == POISON_I).any() and not (buf["images"][1] == POISON_F).any()
    for k in ("gv", "gtex"):
        t = buf[k][1]
        assert torch.isfinite(t).all() and not (t == POISON_F).any()
    assert float(buf["gv"][1].abs().sum()) > 0 and float(buf["gtex"][1].abs().sum()) > 0
    hp = nr.RasterizeHyperparam(image_size=S, anti_aliasing=False)
    img = nr.rasterize_rgba(v, faces, nr.RasterizeParam(textures=tex), hp)
    assert torch.equal(img.reshape(-1), buf["images"][1])


# ---------------------------------------------------------------------------------------------------------------- 6
def test_abi_rejections(nr):
    """NR_FACE_TEXTURES with uv pointers, with an aux map, without NR_DRAW_RGB, with ts < 1 and with oversize cubes is
    refused with NR_ERR_INVALID_ARGUMENT before anything runs."""
    from neural_renderer_v2_pytorch_b200 import _lib
    L = _lib.lib()
    B, S, nf, ts = 1, 16, 2, 2
    v = torch.rand((B, 6, 3), device="cuda")
    faces = torch.arange(6, dtype=torch.int32, device="cuda").reshape(nf, 3)
    tex = torch.rand((B, nf, ts, ts, ts, 3), device="cuda")
    vt = torch.rand((B, 3, 2), device="cuda")
    ft = torch.zeros((nf, 3), dtype=torch.int32, device="cuda")
    fim = torch.empty((B, S, S), dtype=torch.int32, device="cuda")
    img = torch.empty((B, 4, S, S), device="cuda")
    aux = torch.empty((B, S, S, 6), device="cuda")
    ws = torch.empty(1 << 22, dtype=torch.uint8, device="cuda")
    base = (ws.data_ptr() + 255) & ~255
    ptr = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    rgba = _lib.NR_DRAW_RGB | _lib.NR_DRAW_SILHOUETTES | _lib.NR_FACE_TEXTURES

    def forward(flags, ts_=ts, nf_=nf, nvt=0, vt_=None, ft_=None, aux_=None):
        cfg = _config(_lib, B, 6, nf_, S, flags, ts_, nvt)
        return L.nr_rasterize_forward(ctypes.byref(cfg), ptr(v), ptr(faces), ptr(vt_), ptr(ft_), ptr(tex), ptr(fim), None,
                                      None, ptr(img), None, ptr(aux_), None, ctypes.c_void_p(base), 1 << 21, 1024, None,
                                      None, None, None, None)

    assert forward(rgba) == _lib.NR_OK
    torch.cuda.synchronize()
    bad = _lib.NR_ERR_INVALID_ARGUMENT
    assert forward(rgba, vt_=vt) == bad
    assert forward(rgba, ft_=ft) == bad
    assert forward(rgba, nvt=3, vt_=vt, ft_=ft) == bad
    assert forward(rgba, aux_=aux) == bad
    assert forward(_lib.NR_DRAW_SILHOUETTES | _lib.NR_FACE_TEXTURES) == bad
    assert forward(rgba, ts_=0) == bad
    assert forward(rgba, ts_=1 << 10, nf_=nf) == bad                   # nf ts^3 3 >= 2^31
    assert forward(rgba, ts_=1291) == bad
    cfg = _config(_lib, B, 6, nf, S, rgba, ts)
    gv, gt = torch.zeros_like(v), torch.zeros_like(tex)
    args = lambda vt_, ft_, aux_, gvt: (ctypes.byref(cfg), ptr(v), ptr(faces), ptr(vt_), ptr(ft_), ptr(tex), ptr(fim),
                                        ptr(img), ptr(aux_), None, ptr(img), ptr(gv), ptr(gt), ptr(gvt), None, None, None)
    assert L.nr_rasterize_backward(*args(None, None, None, None)) == _lib.NR_OK
    assert L.nr_rasterize_backward(*args(vt, ft, None, None)) == bad
    assert L.nr_rasterize_backward(*args(None, None, aux, None)) == bad
    assert L.nr_rasterize_backward(*args(None, None, None, vt)) == bad
    torch.cuda.synchronize()
    with pytest.raises(AssertionError):
        nr.rasterize_rgb(v, faces, nr.RasterizeParam(vertices_textures=vt, textures=tex),
                         nr.RasterizeHyperparam(image_size=S, anti_aliasing=False))
