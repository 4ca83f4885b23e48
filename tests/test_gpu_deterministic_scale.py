"""Deterministic mode (hyperparams.deterministic) at the sizes of upstream gradient real losses produce.

The deterministic backward sums 64-bit fixed point in units of 2^(E_b - 32), E_b the frexp exponent of view b's
max |grad_images|.  A mean loss over a 64 x 4 x 512^2 image hands the backward G ~ 1e-8, and a loss scaler (AMP)
multiplies it by 2^16 and more: a fixed unit cannot resolve the first and overflows on the second.  Every test
here scales G by powers of two 2^k: float32 products then scale exactly, so a difference comes from the
accumulation, not from the inputs.

Reference: autograd of the oracle pipeline (oracle/pipeline.py, torch on the CPU) with the same scaled G, under the
suite's bar |d| <= 1e-5 |ref| + 1e-5 max|ref| (lit vertex gradients: 1e-4 max|ref|, their normal path goes through
torch's float atomics).  An entry passes within the bar of the float32 oracle or of the same pipeline run in float64:
where G is small the stencil term of the vertex gradients vanishes below its threshold, the scale of the bar drops
with it, and the float32 oracle itself then lies up to 1.1e-5 of the scale from the float64 one on a few entries.
The float-atomic mode is the control at every scale.
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import pipeline as ref

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FIXTURES = ["case_rgba_64", "case_rgb_ortho_aa_32", "case_depth_64", "lit_rgb_48"]
KS = [-40, -30, -26, -20, -14, 0, 16, 24, 30]
# where the threshold guard (assert_guard) finds a stencil difference at the threshold, the nearest clean exponent
SCALES = {f: KS for f in FIXTURES}
SCALES["case_rgb_ortho_aa_32"] = [-40, -30, -26, -20, -11, 0, 16, 24, 30]     # -12 .. -17 fail the guard
SCALES["case_depth_64"] = [-40, -30, -26, -19, -14, 0, 16, 24, 30]            # -20 and -21 fail the guard
LIGHT_KEYS = ("dir_color", "dir_direction", "amb_color", "spec_color", "spec_alpha")
LINEAR = ("grad_textures", "grad_vertices_textures", "grad_vertices_z") + LIGHT_KEYS   # linear in G
STENCIL_EPS = 1e-4      # pipeline.maximum's absolute threshold


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
    return dict(np.load(os.path.join(GOLDEN, name + ".npz")))


def _light_params(d, dev, dtype=torch.float32):
    return {k: torch.from_numpy(d[k].copy()).to(dev, dtype).requires_grad_(True) for k in LIGHT_KEYS}


def _grads(v, tex, vt, P):
    out = {"grad_vertices": v.grad.detach().clone()}
    out["grad_vertices_z"] = out["grad_vertices"][..., 2]
    if tex is not None:
        out["grad_textures"] = tex.grad.detach().clone()
        out["grad_vertices_textures"] = vt.grad.detach().clone()
    for k in P or ():
        out[k] = P[k].grad.detach().clone()
    return out


_ORACLE = {}


def oracle_run(name, k, dtype=torch.float32):
    """Autograd of the oracle pipeline with G * 2^k in `dtype`: every gradient, and the stencil's (right, left) pairs
    at the foreground pixels (internal orientation) for the threshold guard."""
    if (name, k, dtype) in _ORACLE:
        return _ORACLE[name, k, dtype]
    d = _load(name)
    mode = "lit" if name.startswith("lit") else str(d["mode"])
    rgb = mode in ("rgb", "rgba", "lit")
    v = torch.from_numpy(d["vertices"]).to(dtype).requires_grad_(True)
    tex = vt = P = lights = None
    kw = {}
    if rgb:
        tex = torch.from_numpy(d["textures"]).to(dtype).requires_grad_(True)
        vt = torch.from_numpy(d["vertices_textures"]).to(dtype).requires_grad_(True)
        kw = dict(vertices_textures=vt, faces_textures=d["faces_textures"], textures=tex)
    if mode == "lit":
        P = _light_params(d, "cpu", dtype)
        lights = [dict(type="directional", color=P["dir_color"], direction=P["dir_direction"], backside=True),
                  dict(type="ambient", color=P["amb_color"]),
                  dict(type="specular", color=P["spec_color"], alpha=P["spec_alpha"], backside=True)]
    S, aa = int(d["image_size"]), bool(d["anti_aliasing"])
    img, maps = ref.rasterize(v, d["faces"], S, aa, near=float(d["near"]), far=float(d["far"]),
                              draw_backside=bool(d["draw_backside"]), draw_rgb=rgb,
                              draw_silhouettes=mode in ("silhouettes", "rgba"), draw_depth=mode == "depth",
                              lights=lights, return_maps=True, **kw)
    G = torch.from_numpy(d["grad_images"]).to(dtype).reshape(img.shape) * 2.0 ** k
    (img * G).sum().backward()
    # the upstream gradient of the internal image, as the stencil sees it
    x = maps["internal_images"].detach().requires_grad_(True)
    y = torch.flip(x.permute(0, 3, 1, 2), dims=(2, 3))
    if aa:
        y = (y[:, :, 0::2, 0::2] + y[:, :, 1::2, 0::2] + y[:, :, 0::2, 1::2] + y[:, :, 1::2, 1::2]) / 4.
    (y * G).sum().backward()
    out = _grads(v, tex, vt, P)
    out["pairs"] = _stencil_pairs(x.detach(), x.grad, maps["face_index_map"] >= 0)
    _ORACLE[name, k, dtype] = out
    return out


def _stencil_pairs(images, grad, fg):
    """(right, left) of both axes as pipeline.differentiation_backward forms them, at foreground pixels"""
    R = images.shape[1]
    step = 2. / R
    pairs = []
    for ax in (1, 2):
        n = R - 1
        a0, a1 = images.narrow(ax, 0, n), images.narrow(ax, 1, n)
        g0, g1 = grad.narrow(ax, 0, n), grad.narrow(ax, 1, n)
        r = -((a0 - a1) * g1).sum(-1) / step
        l_ = -((a1 - a0) * g0).sum(-1) / step
        pad_lo, pad_hi = [0, 0, 0, 0], [0, 0, 0, 0]
        pad_lo[2 * (2 - ax) + 1], pad_hi[2 * (2 - ax)] = 1, 1
        r = F.pad(r, pad_lo) + F.pad(r, pad_hi)
        l_ = F.pad(l_, pad_hi) + F.pad(l_, pad_lo)
        pairs.append((r[fg], l_[fg]))
    return pairs


def assert_guard(name, k):
    """No stencil difference |r - l| within a relative 1e-3 of the absolute threshold: a last-bit difference between
    kernel and oracle cannot then move a pixel across it."""
    for r, l_ in oracle_run(name, k)["pairs"]:
        d = (r - l_).abs()
        near = ((d - STENCIL_EPS).abs() <= 1e-3 * STENCIL_EPS).sum().item()
        assert near == 0, "%s at 2^%d: %d stencil differences at the 1e-4 threshold" % (name, k, near)


def cuda_run(nr, name, det, G=None, k=0, path="tiles", dev="cuda:0"):
    """One forward + backward of a fixture on the CUDA path with upstream gradient G (default: the fixture's * 2^k);
    every gradient, the image and the call's G."""
    from neural_renderer_v2_pytorch_b200 import rasterize as rz
    d = _load(name)
    lit = name.startswith("lit")
    mode = str(d["mode"])
    t = lambda key: torch.from_numpy(d[key]).to(dev)
    v = t("vertices").requires_grad_(True)
    tex = vt = P = None
    hp = nr.RasterizeHyperparam(image_size=int(d["image_size"]), near=float(d["near"]), far=float(d["far"]),
                                anti_aliasing=bool(d["anti_aliasing"]), draw_backside=bool(d["draw_backside"]))
    hp.deterministic = det
    if mode in ("rgb", "rgba"):
        tex, vt = t("textures").requires_grad_(True), t("vertices_textures").requires_grad_(True)
        lights = None
        if lit:
            P = _light_params(d, dev)
            lights = [nr.DirectionalLight(P["dir_color"], P["dir_direction"], backside=True),
                      nr.AmbientLight(P["amb_color"]), nr.SpecularLight(P["spec_color"], P["spec_alpha"], backside=True)]
        p = nr.RasterizeParam(vertices_textures=vt, faces_textures=t("faces_textures"), textures=tex, lights=lights)
    else:
        p = nr.RasterizeParam()
    fn = {"silhouettes": nr.rasterize_silhouettes, "rgb": nr.rasterize_rgb, "rgba": nr.rasterize_rgba,
          "depth": nr.rasterize_depth}[mode]
    saved = (rz.FORCE_FINE_TILES, rz.FORCE_DENSE_RASTER)
    rz.FORCE_FINE_TILES = path == "fine"
    rz.FORCE_DENSE_RASTER = True if path == "dense" else saved[1]
    try:
        img = fn(v, t("faces"), p, hp)
        if G is None:
            G = t("grad_images") * 2.0 ** k
        img.backward(G)
        torch.cuda.synchronize()
    finally:
        rz.FORCE_FINE_TILES, rz.FORCE_DENSE_RASTER = saved
    out = _grads(v, tex, vt, P)
    out["images"], out["G"] = img.detach(), G
    return out


def _check_against(got, want, want64, name, what=""):
    for key in want:
        if key in ("pairs", "grad_vertices_z"):
            continue
        g, w, w64 = got[key].cpu().numpy().astype(np.float64), want[key].double().numpy(), want64[key].numpy()
        if key == "grad_vertices" and name.startswith("lit"):
            err = np.abs(g - w).max() / np.abs(w).max()
            assert err <= 1e-4, "%s%s: grad_vertices %.3g of the scale" % (name, what, err)
            continue
        bad = np.ones(g.shape, bool)
        for r in (w, w64):
            bad &= np.abs(g - r) > 1e-5 * np.abs(r) + 1e-5 * np.abs(r).max()
        assert not bad.any(), "%s%s: %s: %d / %d beyond the bar of both oracles, max |d| = %.3g (scale %.3g)" % (
            name, what, key, bad.sum(), bad.size, np.abs(g - w64).max(), np.abs(w64).max())


PARAMS = [(f, k, m) for f in FIXTURES for k in SCALES[f] for m in ("deterministic", "float")] + \
         [("case_rgba_64", k, m) for k in KS for m in ("deterministic-fine", "deterministic-dense")]


@pytest.mark.parametrize("fixture,k,mode", PARAMS)
def test_matches_the_oracle_at_every_scale(nr, fixture, k, mode):
    """Every gradient of the fixture at G * 2^k against the oracle's at the same G, 2^-40 .. 2^30: from far below
    the fixed point's old resolution (2^-32) to sums far past its old range (2^31)."""
    assert_guard(fixture, k)
    want = oracle_run(fixture, k)
    if k == max(SCALES[fixture]):
        big = max(float(np.abs(w.numpy()).max()) for key, w in want.items() if key != "pairs")
        assert big > 2.0 ** 31, "%s: 2^%d keeps every |ref| below 2^31 (max %.3g)" % (fixture, k, big)
    det = mode.startswith("deterministic")
    path = mode.split("-")[1] if "-" in mode else "tiles"
    got = cuda_run(nr, fixture, det, k=k, path=path)
    for key in want:
        if key != "pairs":
            assert torch.isfinite(got[key]).all(), key
    # (the oracle's lighting runs in float32 only)
    want64 = want if fixture.startswith("lit") else oracle_run(fixture, k, torch.float64)
    _check_against(got, want, want64, fixture, " at 2^%d (%s)" % (k, mode))


@pytest.mark.parametrize("fixture", ["lit_rgb_48", "case_rgba_64", "case_depth_64"])
def test_power_of_two_scaling_is_exact(nr, fixture):
    """Deterministic: G * 2^k gives exactly 2^k times every gradient that is linear in G; scaling only view 0's G by
    2^-20 leaves every gradient of view 1 bit-identical (xy included) and scales view 0's linear ones exactly."""
    base = cuda_run(nr, fixture, True)
    for k in (-26, 24):
        got = cuda_run(nr, fixture, True, k=k)
        for key in LINEAR:
            if key in base:
                assert torch.equal(got[key], base[key] * 2.0 ** k), "%s: %s at 2^%d is not 2^k times" % (fixture, key, k)
    G = base["G"].clone()
    G[0] *= 2.0 ** -20
    got = cuda_run(nr, fixture, True, G=G)
    for key in base:
        if key in ("images", "G"):
            continue
        # light tensors are [B, ...] like every other gradient here
        assert torch.equal(got[key][1], base[key][1]), "%s: %s of view 1 changed with view 0's scale" % (fixture, key)
        if key in LINEAR:
            assert torch.equal(got[key][0], base[key][0] * 2.0 ** -20), "%s: %s of view 0" % (fixture, key)


def _mean_loss_run(nr, workload, det, inp, target, w):
    dev = torch.device("cuda:0")
    v = inp["vertices"].to(dev).requires_grad_(True)
    tex_p = inp["textures"].to(dev).requires_grad_(True)
    vt = inp["vt"].to(dev).requires_grad_(True)
    hp = nr.RasterizeHyperparam(image_size=w["S"], anti_aliasing=w["aa"])
    hp.deterministic = det
    tex = torch.tanh(tex_p) if w.get("tanh") else tex_p
    p = nr.RasterizeParam(vertices_textures=vt, faces_textures=inp["ft"].to(dev), textures=tex)
    fn = nr.rasterize_rgba if w["mode"] == "rgba" else nr.rasterize_rgb
    F.mse_loss(fn(v, inp["faces"].to(dev), p, hp), target).backward()
    torch.cuda.synchronize()
    return {"grad_vertices": v.grad, "grad_textures": tex_p.grad, "grad_vertices_textures": vt.grad}


@pytest.mark.parametrize("workload", ["cfg2", "cfg5"])
def test_full_size_mean_loss(nr, workload):
    """G of F.mse_loss(image, target) at full size (config 2: 64 views of RGBA at 512^2, G ~ 1e-8; config 5: 32
    anti-aliased RGB views of tanh textures): deterministic gradients within the bar of the float-atomic ones of the
    same call, and bit-identical from run to run."""
    import bench
    dev = torch.device("cuda:0")
    w = dict(bench.WORKLOADS[workload])
    inp = bench.make_inputs(w, 1000, dev, nr)
    # the target: the same scene with every vertex moved a little
    jitter = torch.randn(inp["vertices"].shape, generator=torch.Generator().manual_seed(3)) * 2e-3
    hp = nr.RasterizeHyperparam(image_size=w["S"], anti_aliasing=w["aa"])
    tex = torch.tanh(inp["textures"]) if w.get("tanh") else inp["textures"]
    p = nr.RasterizeParam(vertices_textures=inp["vt"].to(dev), faces_textures=inp["ft"].to(dev), textures=tex.to(dev))
    fn = nr.rasterize_rgba if w["mode"] == "rgba" else nr.rasterize_rgb
    with torch.no_grad():
        target = fn((inp["vertices"] + jitter).to(dev), inp["faces"].to(dev), p, hp)
    flt = _mean_loss_run(nr, workload, False, inp, target, w)
    det = _mean_loss_run(nr, workload, True, inp, target, w)
    det2 = _mean_loss_run(nr, workload, True, inp, target, w)
    for key in flt:
        assert float(flt[key].abs().max()) > 0, key
        grad_close(det[key].cpu().numpy(), flt[key].cpu().numpy(), "%s %s" % (workload, key))
        assert torch.equal(det[key], det2[key]), "%s: %s not bit-reproducible" % (workload, key)


def _same_bits(a, b):
    """torch.equal with NaN equal to NaN"""
    return torch.equal(a.isnan(), b.isnan()) and torch.equal(a.nan_to_num(0., 0., 0.), b.nan_to_num(0., 0., 0.)) and \
        torch.equal(a.isinf(), b.isinf()) and torch.equal(a.sign(), b.sign())


def _masks_equal_and_finite_close(a, b, what):
    for name, f in (("NaN", torch.isnan), ("+inf", lambda x: x == float("inf")), ("-inf", lambda x: x == -float("inf"))):
        assert torch.equal(f(a), f(b)), "%s: %s masks differ (%d vs %d)" % (what, name, int(f(a).sum()), int(f(b).sum()))
    fin = torch.isfinite(b)
    grad_close(a[fin].cpu().numpy(), b[fin].cpu().numpy(), what)


def test_non_finite_upstream_gradient(nr):
    """NaN at a foreground pixel of view 0, +inf and -inf at two neighbouring foreground pixels of one face of view 1
    (they meet on its vertices): every gradient has the same NaN / +inf / -inf entries in deterministic and in float
    mode, the finite entries agree within the bar, and a view's bits do not depend on the other view's G."""
    name = "case_rgba_64"
    d = _load(name)
    G = torch.from_numpy(d["grad_images"]).cuda()
    fim = torch.flip(torch.from_numpy(d["face_index_map"]), dims=(1, 2))     # output orientation [B, S, S]
    ys, xs = torch.nonzero(fim[0] >= 0, as_tuple=True)
    y0, x0 = int(ys[len(ys) // 2]), int(xs[len(xs) // 2])
    # two horizontal neighbours on the same face: +inf and -inf meet on its three vertices
    same = (fim[1] >= 0) & (fim[1] == torch.roll(fim[1], -1, dims=1))
    same[:, -1] = False
    ys, xs = torch.nonzero(same, as_tuple=True)
    y1, x1 = int(ys[len(ys) // 2]), int(xs[len(xs) // 2])
    bad = G.clone()
    bad[0, :, y0, x0] = float("nan")
    bad[1, :3, y1, x1] = float("inf")
    bad[1, :3, y1, x1 + 1] = -float("inf")
    det, flt = cuda_run(nr, name, True, G=bad), cuda_run(nr, name, False, G=bad)
    assert bool(torch.isnan(flt["grad_vertices"][1]).any()), "+inf and -inf did not meet"
    for key in ("grad_vertices", "grad_textures", "grad_vertices_textures"):
        assert not bool(torch.isfinite(flt[key]).all()), key
        _masks_equal_and_finite_close(det[key], flt[key], key)
    # each view against the same call with the other view's non-finite pixels zeroed: bit-identical
    for b in (0, 1):
        clean = bad.clone()
        clean[1 - b] = torch.where(torch.isfinite(bad[1 - b]), bad[1 - b], torch.zeros_like(bad[1 - b]))
        one = cuda_run(nr, name, True, G=clean)
        for key in ("grad_vertices", "grad_textures", "grad_vertices_textures"):
            assert _same_bits(one[key][b], det[key][b]), "view %d: %s" % (b, key)
    zeroed = torch.where(torch.isfinite(bad), bad, torch.zeros_like(bad))
    clean = cuda_run(nr, name, True, G=zeroed)
    for b in (0, 1):
        for key in ("grad_vertices", "grad_textures", "grad_vertices_textures"):
            assert bool(torch.isfinite(clean[key][b]).all()), key


def test_non_finite_vertices_through_the_backward(nr):
    """The z = +inf (and NaN, +-inf x / y) geometry of test_gpu_parity.py::test_non_finite_vertices through the
    backward of both modes: equal NaN / +inf / -inf masks, finite entries within the bar."""
    rng = np.random.RandomState(4)
    c = rng.uniform(-1.1, 1.1, size=(1, 400, 1, 2))
    xy = c + rng.normal(0, 0.3, size=(1, 400, 3, 2))
    z = rng.uniform(1.0, 3.0, size=(1, 400, 1, 1)) + rng.normal(0, 0.02, size=(1, 400, 3, 1))
    f = np.concatenate([xy, z], -1).astype(np.float32)
    f[0, 3, 0, 0] = np.nan
    f[0, 9, 1, 1] = np.inf
    f[0, 15, 2, 0] = -np.inf
    f[0, 21, 0, 2] = np.nan
    f[0, 27, 1, 2] = np.inf
    f[0, 33, 2, 2] = 0.0
    f[0, 39, :, 2] = -1.0
    R = 96
    faces = torch.arange(1200, dtype=torch.int32).reshape(400, 3).cuda()
    G = torch.randn((1, 2, R, R), generator=torch.Generator().manual_seed(9)).cuda()
    out = {}
    for det in (True, False):
        v = torch.from_numpy(f).reshape(1, 1200, 3).cuda().requires_grad_(True)
        hp = nr.RasterizeHyperparam(image_size=R, anti_aliasing=False, draw_rgb=False, draw_silhouettes=True,
                                    draw_depth=True)
        hp.deterministic = det
        img = nr.rasterize_core(v, faces, nr.RasterizeParam(), hp)
        img.backward(G.reshape(img.shape))
        torch.cuda.synchronize()
        out[det] = v.grad
    _masks_equal_and_finite_close(out[True], out[False], "grad_vertices")


def test_capture_step_picks_up_a_new_scale(nr):
    """A deterministic step captured with nr.capture_step; the loss weight changes in place between replays
    (1, 2^-26, 2^24): each replay equals the eager step with that weight bit for bit, so the fixed-point scale is
    chosen on the device at every replay, not on the host or at capture."""
    d = _load("lit_rgb_48")
    dev = "cuda:0"
    t = lambda key: torch.from_numpy(d[key]).to(dev)
    v, tex, vt = t("vertices").requires_grad_(True), t("textures").requires_grad_(True), t("vertices_textures").requires_grad_(True)
    P = _light_params(d, dev)
    G, weight = t("grad_images"), torch.ones((), device=dev)
    faces, ft = t("faces"), t("faces_textures")
    params = [v, tex, vt] + [P[k] for k in LIGHT_KEYS]

    def step():
        hp = nr.RasterizeHyperparam(image_size=int(d["image_size"]), anti_aliasing=bool(d["anti_aliasing"]),
                                    draw_backside=bool(d["draw_backside"]))
        hp.deterministic = True
        lights = [nr.DirectionalLight(P["dir_color"], P["dir_direction"], backside=True),
                  nr.AmbientLight(P["amb_color"]), nr.SpecularLight(P["spec_color"], P["spec_alpha"], backside=True)]
        p = nr.RasterizeParam(vertices_textures=vt, faces_textures=ft, textures=tex, lights=lights)
        img = nr.rasterize_rgb(v, faces, p, hp)
        (img * G * weight).sum().backward()
        return img

    def eager():
        for q in params:
            q.grad = None
        step()
        torch.cuda.synchronize()
        return [q.grad.clone() for q in params]

    replay = nr.capture_step(step, params=params, warmup=2)
    static = [q.grad for q in params]      # the replayed backward writes these; eager steps make new ones
    for s in (1.0, 2.0 ** -26, 2.0 ** 24):
        weight.fill_(s)
        replay()
        torch.cuda.synchronize()
        got = [g.clone() for g in static]
        want = eager()
        for i, (a, b) in enumerate(zip(got, want)):
            assert torch.equal(a, b), "weight %g: gradient of parameter %d differs from the eager step" % (s, i)
