"""Gradients with respect to the lights (color, direction, alpha) from the fused backward, against autograd of the
oracle's torch-op lighting (oracle/pipeline.py::light_color_weights, rasterize.py:252-283), on every raster path.

Bar for the light gradients: |d| <= 1e-5 * |ref| + 1e-5 * max|ref| per tensor, as for every other gradient
(test_gpu_parity.py::grad_close).  Asking for light gradients must not change anything else: the images are
bit-identical to the same call with constant lights, and the vertex / texture gradients agree with it."""
import os

import numpy as np
import pytest
import torch

from oracle import pipeline as ref

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FIXTURES = ["lit_rgb_48", "lit_rgb_aa_24"]
LIGHT_KEYS = ("dir_color", "dir_direction", "amb_color", "spec_color", "spec_alpha")


@pytest.fixture(scope="module")
def nr():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import neural_renderer_v2_pytorch_b200 as nr_
    return nr_


def grad_close(got, want, what):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    scale = np.abs(want).max()
    tol = 1e-5 * np.abs(want) + 1e-5 * scale
    bad = np.abs(got - want) > tol
    assert not bad.any(), "%s: %d / %d beyond tolerance, max |d| = %.3g (scale %.3g)" % (
        what, bad.sum(), bad.size, np.abs(got - want).max(), scale)


def _load(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def _light_params(d, dev, grad, which=LIGHT_KEYS):
    """The fixture's light tensors on `dev`, fresh leaves (requiring grad when `grad`)."""
    return {k: torch.from_numpy(d[k].copy()).to(dev).requires_grad_(grad and k in which) for k in LIGHT_KEYS}


def _lights(nr, P, lb, kinds="das"):
    out = []
    if "d" in kinds:
        out.append(nr.DirectionalLight(P["dir_color"], P["dir_direction"], backside=lb))
    if "a" in kinds:
        out.append(nr.AmbientLight(P["amb_color"]))
    if "s" in kinds:
        out.append(nr.SpecularLight(P["spec_color"], P["spec_alpha"], backside=lb))
    return out


def _oracle_lights(P, lb, kinds="das"):
    out = []
    if "d" in kinds:
        out.append(dict(type="directional", color=P["dir_color"], direction=P["dir_direction"], backside=lb))
    if "a" in kinds:
        out.append(dict(type="ambient", color=P["amb_color"]))
    if "s" in kinds:
        out.append(dict(type="specular", color=P["spec_color"], alpha=P["spec_alpha"], backside=lb))
    return out


_ORACLE = {}


def oracle_grads(name, lb, kinds="das"):
    """Autograd of the oracle pipeline (CPU, torch ops) with respect to every light tensor."""
    key = (name, lb, kinds)
    if key not in _ORACLE:
        d = _load(name)
        P = _light_params(d, "cpu", True)
        img = ref.rasterize(torch.from_numpy(d["vertices"]), d["faces"], int(d["image_size"]), bool(d["anti_aliasing"]),
                            near=float(d["near"]), far=float(d["far"]), draw_backside=bool(d["draw_backside"]),
                            draw_rgb=True, draw_silhouettes=False,
                            vertices_textures=torch.from_numpy(d["vertices_textures"]), faces_textures=d["faces_textures"],
                            textures=torch.from_numpy(d["textures"]), lights=_oracle_lights(P, lb, kinds))
        (img * torch.from_numpy(d["grad_images"])).sum().backward()
        _ORACLE[key] = {k: P[k].grad.numpy().copy() for k in LIGHT_KEYS if P[k].grad is not None}
    return _ORACLE[key]


def render(nr, d, lights, grad_mesh=True, deterministic=False, dev="cuda:0"):
    t = lambda k: torch.from_numpy(d[k]).to(dev)
    v = t("vertices").requires_grad_(grad_mesh)
    tex = t("textures").requires_grad_(grad_mesh)
    hp = nr.RasterizeHyperparam(image_size=int(d["image_size"]), anti_aliasing=bool(d["anti_aliasing"]),
                                draw_backside=bool(d["draw_backside"]), near=float(d["near"]), far=float(d["far"]))
    hp.deterministic = deterministic
    p = nr.RasterizeParam(vertices_textures=t("vertices_textures"), faces_textures=t("faces_textures"), textures=tex,
                          lights=lights)
    images = nr.rasterize_rgb(v, t("faces"), p, hp)
    if images.requires_grad:
        (images * t("grad_images")).sum().backward()
    torch.cuda.synchronize()
    return images.detach(), v, tex


class _Mode:
    """Raster path switches of rasterize.py, set for the duration of a test.  The vertex normals are summed in a
    fixed order (lights.vertex_normals(deterministic=True)) in every mode: by default they come from torch's index_add,
    whose float atomics make two lit forwards differ in the last bits, and the test compares two forwards bit for bit
    to show that asking for light gradients leaves the forward untouched."""

    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        from neural_renderer_v2_pytorch_b200 import rasterize as rz
        self.rz, self.saved = rz, (rz.FORCE_FINE_TILES, rz.FORCE_DENSE_RASTER, rz.USE_AUX_MAP)
        self.normals = rz.light_lib.vertex_normals
        normals = self.normals
        rz.light_lib.vertex_normals = lambda v, f, deterministic=False: normals(v, f, deterministic=True)
        if self.mode == "fine":
            rz.FORCE_FINE_TILES = True
        elif self.mode == "dense":
            rz.FORCE_DENSE_RASTER = True
        elif self.mode == "aux":
            rz.USE_AUX_MAP = True
        return self

    def __exit__(self, *exc):
        self.rz.FORCE_FINE_TILES, self.rz.FORCE_DENSE_RASTER, self.rz.USE_AUX_MAP = self.saved
        self.rz.light_lib.vertex_normals = self.normals


@pytest.mark.parametrize("mode", ["tiles", "fine", "dense", "aux", "deterministic"])
@pytest.mark.parametrize("lb", [False, True])
@pytest.mark.parametrize("name", FIXTURES)
def test_light_gradients_match_the_oracle(nr, name, lb, mode):
    """All three light types, every light tensor requiring grad, AA off / on (the two fixtures), backside off / on,
    on the 16x16 tile path, 8x8 tiles, the dense z-buffer path, with the aux map and in deterministic mode."""
    d = _load(name)
    det = mode == "deterministic"
    with _Mode(mode):
        img0, v0, tex0 = render(nr, d, _lights(nr, _light_params(d, "cuda:0", False), lb), deterministic=det)
        P = _light_params(d, "cuda:0", True)
        img1, v1, tex1 = render(nr, d, _lights(nr, P, lb), deterministic=det)
        if det:
            P2 = _light_params(d, "cuda:0", True)
            render(nr, d, _lights(nr, P2, lb), deterministic=True)
    assert torch.equal(img0, img1), "light gradients changed the image"
    grad_close(tex1.grad.cpu().numpy(), tex0.grad.cpu().numpy(), "grad_textures")
    gv1, gv0 = v1.grad.cpu().numpy(), v0.grad.cpu().numpy()
    assert np.abs(gv1 - gv0).max() <= 1e-4 * np.abs(gv0).max()
    want = oracle_grads(name, lb)
    for k in LIGHT_KEYS:
        got = P[k].grad
        assert got is not None and got.dtype == torch.float32 and got.shape == P[k].shape, k
        assert torch.isfinite(got).all(), k
        grad_close(got.cpu().numpy(), want[k], k)
        if det:
            assert torch.equal(got, P2[k].grad), "%s: deterministic mode is not bit-reproducible" % k


@pytest.mark.parametrize("name", FIXTURES)
def test_only_the_lights_require_grad(nr, name):
    """vertices and textures constant: the backward still runs and fills the light gradients"""
    d = _load(name)
    lb = bool(d["light_backside"])
    P = _light_params(d, "cuda:0", True)
    _, v, tex = render(nr, d, _lights(nr, P, lb), grad_mesh=False)
    assert v.grad is None and tex.grad is None
    want = oracle_grads(name, lb)
    for k in LIGHT_KEYS:
        grad_close(P[k].grad.cpu().numpy(), want[k], k)


@pytest.mark.parametrize("name", FIXTURES)
def test_shared_light_gradient_is_the_sum_over_views(nr, name):
    """one light for all views: Parameter [1,3] passed as .expand(B, 3) (colour and direction)"""
    d = dict(_load(name))
    B = d["vertices"].shape[0]
    for k in LIGHT_KEYS:            # every view gets view 0's light
        d[k] = np.ascontiguousarray(np.repeat(d[k][:1], B, axis=0))
    lb = bool(d["light_backside"])
    dev = "cuda:0"
    dc = torch.nn.Parameter(torch.from_numpy(d["dir_color"][:1]).to(dev))
    dd = torch.nn.Parameter(torch.from_numpy(d["dir_direction"][:1]).to(dev))
    ac = torch.nn.Parameter(torch.from_numpy(d["amb_color"][:1]).to(dev))
    lights = [nr.DirectionalLight(dc.expand(B, 3), dd.expand(B, 3), backside=lb), nr.AmbientLight(ac.expand(B, 3))]
    render(nr, d, lights)
    P = _light_params(d, "cpu", True)
    img = ref.rasterize(torch.from_numpy(d["vertices"]), d["faces"], int(d["image_size"]), bool(d["anti_aliasing"]),
                        near=float(d["near"]), far=float(d["far"]), draw_backside=bool(d["draw_backside"]),
                        draw_rgb=True, draw_silhouettes=False,
                        vertices_textures=torch.from_numpy(d["vertices_textures"]), faces_textures=d["faces_textures"],
                        textures=torch.from_numpy(d["textures"]), lights=_oracle_lights(P, lb, "da"))
    (img * torch.from_numpy(d["grad_images"])).sum().backward()
    assert dc.grad.shape == (1, 3)
    grad_close(dc.grad.cpu().numpy(), P["dir_color"].grad.sum(0, keepdim=True).numpy(), "shared dir_color")
    grad_close(dd.grad.cpu().numpy(), P["dir_direction"].grad.sum(0, keepdim=True).numpy(), "shared dir_direction")
    grad_close(ac.grad.cpu().numpy(), P["amb_color"].grad.sum(0, keepdim=True).numpy(), "shared amb_color")


def test_specular_alpha_where_the_base_is_zero(nr):
    """A specular light without backside on a view that shows back faces: some lit pixels have a = relu(-n_z) = 0,
    where torch's pow backward gives d alpha = 0 (not NaN)."""
    name = "lit_rgb_48"
    d = _load(name)
    v = torch.from_numpy(d["vertices"])
    fidx = torch.as_tensor(d["faces"]).long()
    _, maps = ref.rasterize(v, d["faces"], int(d["image_size"]), False, draw_backside=bool(d["draw_backside"]),
                            return_maps=True)
    fim, wmap = maps["face_index_map"], maps["weight_map"]
    raw = -ref.compute_normal_map(v, fidx, v[:, fidx], fim, wmap)[..., 2]
    assert int(((raw <= 0) & (fim >= 0)).sum()) > 0 and int(((raw > 0) & (fim >= 0)).sum()) > 0
    P = _light_params(d, "cuda:0", True)
    render(nr, d, _lights(nr, P, False, "s"))
    want = oracle_grads(name, False, "s")
    for k in ("spec_color", "spec_alpha"):
        assert torch.isfinite(P[k].grad).all() and np.isfinite(want[k]).all()
        grad_close(P[k].grad.cpu().numpy(), want[k], k)


@pytest.mark.parametrize("k", [-26, 0, 24])
@pytest.mark.parametrize("deterministic", [False, True])
def test_full_size_ambient_colour_gradient(nr, deterministic, k):
    """Teapot, 64 views at 512^2, RGB, one ambient light: the image is linear in its colour, so
    d loss / d colour[b, c] = sum G * image_unlit[b, c] (float64 sum of an unlit render of the same inputs).  Every
    foreground pixel of a view adds to the same 3 values: the reduction at full contention.  G is uniform in [0, 1)
    so that the sum is well conditioned and the bar measures the reduction, not float32 cancellation.  G is scaled
    by 2^k: 2^-26 is a mean loss over config 2's image, 2^24 a loss scaler's factor that puts the sums past 2^31."""
    import bench
    dev = torch.device("cuda:0")
    w = dict(bench.WORKLOADS["cfg2"], mode="rgb")
    inp = bench.make_inputs(w, 1000, dev, nr)
    B, S = w["views"], w["S"]
    v, faces = inp["vertices"].to(dev), inp["faces"].to(dev)
    vt, ft, tex = inp["vt"].to(dev), inp["ft"].to(dev), inp["textures"].to(dev)
    G = (torch.rand((B, 3, S, S), generator=torch.Generator().manual_seed(5)) * 2.0 ** k).to(dev)

    def hp():
        h = nr.RasterizeHyperparam(image_size=S, anti_aliasing=False)
        h.deterministic = deterministic
        return h

    unlit = nr.rasterize_rgb(v, faces, nr.RasterizeParam(vertices_textures=vt, faces_textures=ft, textures=tex), hp())
    color = (0.5 + torch.rand((B, 3), generator=torch.Generator().manual_seed(6))).to(dev).requires_grad_(True)
    p = nr.RasterizeParam(vertices_textures=vt, faces_textures=ft, textures=tex, lights=[nr.AmbientLight(color)])
    img = nr.rasterize_rgb(v, faces, p, hp())
    (img * G).sum().backward()
    want = (G.double() * unlit.double()).sum(dim=(2, 3))
    if k == 24:
        assert float(want.abs().max()) > 2.0 ** 31
    np.testing.assert_allclose(color.grad.double().cpu().numpy(), want.cpu().numpy(), rtol=1e-5)


@pytest.mark.parametrize("deterministic", [False, True])
def test_capture_step_with_light_parameters(nr, deterministic):
    """A lit step whose light tensors require grad, captured with nr.capture_step: the replayed light gradients equal
    the eager ones (bit for bit in deterministic mode)."""
    d = _load("lit_rgb_48")
    lb = bool(d["light_backside"])
    dev = "cuda:0"
    t = lambda k: torch.from_numpy(d[k]).to(dev)
    v, tex, faces, vt, ft, G = t("vertices").requires_grad_(True), t("textures").requires_grad_(True), t("faces"), \
        t("vertices_textures"), t("faces_textures"), t("grad_images")
    P = _light_params(d, dev, True)
    params = [v, tex] + [P[k] for k in LIGHT_KEYS]

    def step():
        hp = nr.RasterizeHyperparam(image_size=int(d["image_size"]), anti_aliasing=bool(d["anti_aliasing"]),
                                    draw_backside=bool(d["draw_backside"]))
        hp.deterministic = deterministic
        p = nr.RasterizeParam(vertices_textures=vt, faces_textures=ft, textures=tex, lights=_lights(nr, P, lb))
        img = nr.rasterize_rgb(v, faces, p, hp)
        (img * G).sum().backward()
        return img

    for q in params:
        q.grad = None
    step()
    torch.cuda.synchronize()
    eager = {k: P[k].grad.clone() for k in LIGHT_KEYS}
    replay = nr.capture_step(step, params=params, warmup=2)
    for _ in range(2):
        replay()
    torch.cuda.synchronize()
    for k in LIGHT_KEYS:
        if deterministic:
            assert torch.equal(P[k].grad, eager[k]), k
        else:
            grad_close(P[k].grad.cpu().numpy(), eager[k].cpu().numpy(), k)
