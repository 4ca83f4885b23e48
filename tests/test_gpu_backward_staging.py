"""The staged front of k_backward (face indices, stencil image and upstream gradient copied into shared memory by TMA,
csrc/nr_backward.cu) against the unstaged path it replaces (NR_FORCE_UNSTAGED_BACKWARD=1), on the same inputs.

Both paths read the same values and run the same arithmetic, so in deterministic mode (64-bit fixed-point sums) every
gradient is bit-identical between them.  With float atomics the sums are taken in arrival order: the gradients agree
at the suite's bar, |d| <= 1e-5 * |ref| + 1e-5 * max|ref|, and the images are identical (the forward is untouched)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FORCE = "NR_FORCE_UNSTAGED_BACKWARD"


@pytest.fixture(scope="module")
def nr():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import neural_renderer_v2_pytorch_b200 as nr_
    return nr_


@pytest.fixture
def raster_path():
    """Sets rasterize.py's path switches for one test and restores them."""
    from neural_renderer_v2_pytorch_b200 import rasterize as rz
    saved = (rz.FORCE_FINE_TILES, rz.FORCE_DENSE_RASTER)

    def set_path(path):
        rz.FORCE_FINE_TILES = path == "fine"
        rz.FORCE_DENSE_RASTER = True if path == "dense" else saved[1]

    yield set_path
    rz.FORCE_FINE_TILES, rz.FORCE_DENSE_RASTER = saved


def grad_close(got, want, what):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    scale = np.abs(want).max()
    tol = 1e-5 * np.abs(want) + 1e-5 * scale
    bad = np.abs(got - want) > tol
    assert not bad.any(), "%s: %d / %d beyond tolerance, max |d| = %.3g (scale %.3g)" % (
        what, bad.sum(), bad.size, np.abs(got - want).max(), scale)


def both_paths(monkeypatch, run):
    """run() -> dict of tensors, once on the staged path and once forced onto the unstaged one"""
    monkeypatch.delenv(FORCE, raising=False)
    staged = run()
    monkeypatch.setenv(FORCE, "1")
    unstaged = run()
    monkeypatch.delenv(FORCE)
    return staged, unstaged


def compare(staged, unstaged, deterministic):
    assert staged.keys() == unstaged.keys()
    for k in staged:
        a, b = staged[k], unstaged[k]
        assert a is not None and b is not None, k
        if deterministic or k == "images":
            assert torch.equal(a, b), "%s differs between the staged and the unstaged backward" % k
        else:
            grad_close(a.cpu().numpy(), b.cpu().numpy(), k)


def bench_run(nr, workload, deterministic, views=None, S=None, aa=None, mode=None, grad_vt=True, grad_images=None):
    """One forward + backward of a bench.py workload (optionally resized); returns the images and every gradient."""
    import bench
    dev = torch.device("cuda:0")
    w = dict(bench.WORKLOADS[workload])
    if views:
        w["views"] = views
    if S:
        w["S"] = S
    if mode:
        w["mode"] = mode
    if aa is not None:
        w["aa"] = aa
    inp = bench.make_inputs(w, 1000, dev, nr)
    rgb = w["mode"] in ("rgb", "rgba")

    def run():
        v = inp["vertices"].to(dev).requires_grad_(True)
        hp = nr.RasterizeHyperparam(image_size=w["S"], anti_aliasing=w["aa"])
        hp.deterministic = deterministic
        out = {}
        if rgb:
            vt = inp["vt"].to(dev).requires_grad_(grad_vt)
            tex = inp["textures"].to(dev).requires_grad_(True)
            p = nr.RasterizeParam(vertices_textures=vt, faces_textures=inp["ft"].to(dev), textures=tex)
            fn = nr.rasterize_rgba if w["mode"] == "rgba" else nr.rasterize_rgb
        else:
            p = nr.RasterizeParam()
            fn = nr.rasterize_silhouettes
        img = fn(v, inp["faces"].to(dev), p, hp)
        G = inp["G"].to(dev) if grad_images is None else grad_images(inp["G"].to(dev))
        img.backward(G)
        torch.cuda.synchronize()
        out["images"] = img.detach()
        out["grad_vertices"] = v.grad
        if rgb:
            out["grad_textures"] = tex.grad
            if grad_vt:
                out["grad_vertices_textures"] = vt.grad
        return out

    return run


@pytest.mark.parametrize("deterministic", [True, False])
def test_config2_full_size(nr, monkeypatch, deterministic):
    """Config 2 as bench.py runs it: teapot, 64 views at 512^2, RGBA (float mode: the C = 4 variant); in
    deterministic mode also with the gradient of vertices_textures."""
    run = bench_run(nr, "cfg2", deterministic, grad_vt=deterministic)
    compare(*both_paths(monkeypatch, run), deterministic)


@pytest.mark.parametrize("deterministic", [True, False])
def test_anti_aliasing(nr, monkeypatch, deterministic):
    """Config 5's shape (512^2 with 2x anti-aliasing, RGB, orthographic): the upstream gradient is staged from the
    half-resolution box."""
    run = bench_run(nr, "cfg5", deterministic, views=8)
    compare(*both_paths(monkeypatch, run), deterministic)


@pytest.mark.parametrize("path", ["tiles", "fine", "dense"])
@pytest.mark.parametrize("mode", ["rgba", "silhouettes"])
def test_raster_paths(nr, monkeypatch, raster_path, path, mode):
    """Behind the 16x16 tile lists, the 8x8 tiles (the backward then walks every tile) and the dense z-buffer path;
    colour and silhouettes only."""
    raster_path(path)
    run = bench_run(nr, "cfg2", True, views=8, mode=mode)
    compare(*both_paths(monkeypatch, run), True)


@pytest.mark.parametrize("S,aa", [(200, False), (100, True), (202, False), (250, False)])
def test_image_size_not_a_multiple_of_16(nr, monkeypatch, S, aa):
    """Partial tiles at the image border (R % 16 != 0: staged, TMA's zero fill never reaches the stencil), and row
    strides TMA cannot address (R % 4 != 0: both runs take the unstaged path)."""
    run = bench_run(nr, "cfg2", True, views=4, S=S, aa=aa)
    compare(*both_paths(monkeypatch, run), True)


def test_misaligned_grad_images(nr, monkeypatch):
    """A grad_images view whose storage starts 4 bytes past a 16-byte boundary cannot be a TMA source: the backward
    takes the unstaged path and computes what it computes from an aligned copy."""
    def shifted(G):
        buf = torch.empty(G.numel() + 1, device=G.device)
        view = buf[1:].view(G.shape)
        view.copy_(G)
        assert view.is_contiguous() and view.data_ptr() % 16 == 4
        return view

    aligned = bench_run(nr, "cfg2", True, views=4)()
    staged, unstaged = both_paths(monkeypatch, bench_run(nr, "cfg2", True, views=4, grad_images=shifted))
    compare(staged, unstaged, True)
    compare(staged, aligned, True)


@pytest.mark.parametrize("name", ["lit_rgb_48", "lit_rgb_aa_24"])
def test_lit_with_light_gradients(nr, monkeypatch, name):
    """Lights whose colour, direction and exponent require grad (the LGRAD variants), with and without
    anti-aliasing: the light gradients and the gradient of the vertex normals too."""
    d = np.load(os.path.join(GOLDEN, name + ".npz"))
    dev = "cuda:0"
    t = lambda k: torch.from_numpy(d[k]).to(dev)
    lb = bool(d["light_backside"])

    def run():
        v, tex, vt = t("vertices").requires_grad_(True), t("textures").requires_grad_(True), t("vertices_textures").requires_grad_(True)
        P = {k: t(k).requires_grad_(True) for k in ("dir_color", "dir_direction", "amb_color", "spec_color", "spec_alpha")}
        lights = [nr.DirectionalLight(P["dir_color"], P["dir_direction"], backside=lb), nr.AmbientLight(P["amb_color"]),
                  nr.SpecularLight(P["spec_color"], P["spec_alpha"], backside=lb)]
        hp = nr.RasterizeHyperparam(image_size=int(d["image_size"]), anti_aliasing=bool(d["anti_aliasing"]),
                                    draw_backside=bool(d["draw_backside"]), near=float(d["near"]), far=float(d["far"]))
        hp.deterministic = True
        p = nr.RasterizeParam(vertices_textures=vt, faces_textures=t("faces_textures"), textures=tex, lights=lights)
        img = nr.rasterize_rgb(v, t("faces"), p, hp)
        (img * t("grad_images")).sum().backward()
        torch.cuda.synchronize()
        out = dict(images=img.detach(), grad_vertices=v.grad, grad_textures=tex.grad, grad_vertices_textures=vt.grad)
        out.update({"grad_" + k: P[k].grad for k in P})
        return out

    compare(*both_paths(monkeypatch, run), True)
