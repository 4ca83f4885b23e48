"""Differentiable lights on the host side (no GPU): lights.pack_lights keeps light tensors that require grad
connected to the packed [L,B,8] light data, the new C entry point is declared and validates its arguments, and the
closed-form light gradient the backward kernel sums (csrc/nr_backward.cu::light_param_grads) agrees with autograd
of the oracle's torch-op lighting (rasterize.py:252-283)."""
import ctypes

import numpy as np
import torch

import neural_renderer_v2_pytorch_b200 as nr
from neural_renderer_v2_pytorch_b200.lights import pack_lights
from oracle import pipeline as ref


def _lights(B, g):
    r = lambda *s: torch.rand(*s, generator=g)
    lights = [nr.DirectionalLight(r(B, 3).requires_grad_(True), (r(B, 3) - 0.5).requires_grad_(True), backside=True),
              nr.AmbientLight(r(B, 3).requires_grad_(True)),
              nr.SpecularLight(r(B, 3).requires_grad_(True), (1 + r(B)).requires_grad_(True))]
    return lights


def test_pack_lights_accepts_tensors_that_require_grad():
    B = 3
    lights = _lights(B, torch.Generator().manual_seed(0))
    types, data = pack_lights(lights, B, "cpu")
    assert types.tolist() == [1 | 4, 0, 2] and data.shape == (3, B, 8) and data.requires_grad
    assert torch.equal(data[0, :, 0:3], lights[0].color) and torch.equal(data[0, :, 3:6], lights[0].direction)
    assert torch.equal(data[2, :, 6], lights[2].alpha) and torch.equal(data[1, :, 3:8], torch.zeros(B, 5))


def test_pack_lights_routes_each_slot_to_its_tensor():
    """backward of (data * w).sum() puts w's colour / direction / alpha slots into the right .grad; the specular
    direction (the fixed eye vector) and the unused slot feed nothing."""
    B = 2
    lights = _lights(B, torch.Generator().manual_seed(1))
    _, data = pack_lights(lights, B, "cpu")
    w = torch.randn(data.shape, generator=torch.Generator().manual_seed(2))
    (data * w).sum().backward()
    d, a, s = lights
    assert torch.equal(d.color.grad, w[0, :, 0:3]) and torch.equal(d.direction.grad, w[0, :, 3:6])
    assert torch.equal(a.color.grad, w[1, :, 0:3])
    assert torch.equal(s.color.grad, w[2, :, 0:3]) and torch.equal(s.alpha.grad, w[2, :, 6])


def test_shared_light_sums_over_the_views():
    """a light shared by all views is passed as param.expand(B, 3): its gradient is the sum over the views"""
    B = 4
    c = torch.nn.Parameter(torch.rand(1, 3))
    dr = torch.nn.Parameter(torch.rand(1, 3))
    _, data = pack_lights([nr.DirectionalLight(c.expand(B, 3), dr.expand(B, 3))], B, "cpu")
    w = torch.randn(data.shape, generator=torch.Generator().manual_seed(3))
    (data * w).sum().backward()
    assert torch.allclose(c.grad, w[0, :, 0:3].sum(0, keepdim=True))
    assert torch.allclose(dr.grad, w[0, :, 3:6].sum(0, keepdim=True))


def test_pack_lights_dtype_and_constant_lights_unchanged():
    B = 2
    col = torch.rand(B, 3, dtype=torch.float64, requires_grad=True)
    _, data = pack_lights([nr.AmbientLight(col)], B, "cpu")
    assert data.dtype == torch.float32
    data.sum().backward()
    assert col.grad.dtype == torch.float64 and torch.equal(col.grad, torch.ones(B, 3, dtype=torch.float64))
    t1, d1 = pack_lights([nr.AmbientLight(torch.rand(B, 3))], B, "cpu")
    t2, _ = pack_lights([nr.AmbientLight(torch.rand(B, 3))], B, "cpu")
    assert not d1.requires_grad and t1 is t2            # the type tensor is made once per (types, device)
    _, black = pack_lights([], B, "cpu")
    assert torch.equal(black, torch.zeros(1, B, 8))


def test_backward_lights_entry_point_validates_before_any_cuda_call():
    from neural_renderer_v2_pytorch_b200 import _lib
    _lib.build()
    L = _lib.lib()
    assert "nr_rasterize_backward_lights" in _lib.SYMBOLS
    cfg = _lib.RasterConfig(batch=2, num_vertices=3, num_faces=1, image_size=8, flags=_lib.NR_DRAW_RGB,
                            near_plane=0.1, far_plane=100., eps=1e-5, depth_min_delta=1e-4, num_tex_vertices=3,
                            tex_height=2, tex_width=2)
    rc = L.nr_rasterize_backward_lights(ctypes.byref(cfg), *([None] * 14), None, None, None, None)
    assert rc == _lib.NR_ERR_INVALID_ARGUMENT and b"NULL" in L.nr_last_error()


def _closed_form(n, w, light):
    """The kernel's per-pixel light gradient (nr_backward.cu::light_param_grads) in float64 numpy:
    n [P,3] interpolated normals, w [P,3] d loss / d colour weight -> gradient of [colour 3, direction 3, alpha]."""
    kind = light["type"]
    color = light["color"][0].detach().numpy().astype(np.float64)
    out = np.zeros(7)
    if kind == "ambient":
        out[0:3] = w.sum(0)
        return out
    d = light["direction"][0].detach().numpy().astype(np.float64) if kind == "directional" else np.array([0., 0., 1.])
    raw = -(n @ d)
    if light.get("backside"):
        a, gate = np.abs(raw), np.sign(raw)
    else:
        a, gate = np.maximum(raw, 0.), (raw > 0).astype(np.float64)
    s = w @ color
    if kind == "directional":
        out[0:3] = (w * a[:, None]).sum(0)
        out[3:6] = -((s * gate)[:, None] * n).sum(0)
    else:
        alpha = float(light["alpha"][0].detach())
        inten = a ** alpha
        out[0:3] = (w * inten[:, None]).sum(0)
        with np.errstate(divide="ignore"):
            out[6] = np.where(a > 0, s * inten * np.log(np.where(a > 0, a, 1.)), 0.).sum()
    return out


def test_closed_form_matches_autograd_of_the_oracle_lighting():
    """Including normals with a = 0 (relu gate closed, n = 0 background-like pixels): the alpha gradient there is 0,
    like torch's pow backward at a zero base, and never NaN."""
    g = torch.Generator().manual_seed(4)
    P = 400
    n = torch.nn.functional.normalize(torch.randn(1, P, 1, 3, generator=g), dim=-1)
    n[0, :40] = 0.                                                   # a = 0 exactly
    w = torch.randn(1, P, 1, 3, generator=g)
    for backside in (False, True):
        lights = [dict(type="directional", color=torch.rand(1, 3, generator=g).requires_grad_(True),
                       direction=torch.randn(1, 3, generator=g).requires_grad_(True), backside=backside),
                  dict(type="ambient", color=torch.rand(1, 3, generator=g).requires_grad_(True)),
                  dict(type="specular", color=torch.rand(1, 3, generator=g).requires_grad_(True),
                       alpha=(1 + 3 * torch.rand(1, generator=g)).requires_grad_(True), backside=backside)]
        (ref.light_color_weights(n, lights) * w).sum().backward()
        nn_, ww = n[0, :, 0].double().numpy(), w[0, :, 0].double().numpy()
        for L in lights:
            got = _closed_form(nn_, ww, L)
            assert np.all(np.isfinite(got))
            np.testing.assert_allclose(got[0:3], L["color"].grad[0].numpy(), rtol=1e-5, atol=1e-5)
            if L["type"] == "directional":
                np.testing.assert_allclose(got[3:6], L["direction"].grad[0].numpy(), rtol=1e-5, atol=1e-5)
            if L["type"] == "specular":
                assert torch.isfinite(L["alpha"].grad).all()
                np.testing.assert_allclose(got[6], L["alpha"].grad[0].item(), rtol=1e-5, atol=1e-5)


def test_deterministic_vertex_normals_equal_the_index_add_ones():
    """the fixed-order sum of deterministic mode gives the normals of the index_add path, and is differentiable"""
    from neural_renderer_v2_pytorch_b200.lights import vertex_normals
    g = torch.Generator().manual_seed(5)
    v = torch.randn(2, 9, 3, generator=g, requires_grad=True)
    f = torch.tensor([[0, 1, 2], [2, 3, 4], [4, 5, 6], [0, 2, 4], [1, 1, 3], [6, 7, 8], [8, 8, 8]], dtype=torch.int32)
    a, b = vertex_normals(v, f), vertex_normals(v, f, deterministic=True)
    assert torch.allclose(a, b, atol=1e-6)
    ga, = torch.autograd.grad((a * a.detach()).sum(), v)
    gb, = torch.autograd.grad((b * a.detach()).sum(), v)
    assert torch.allclose(ga, gb, atol=1e-5)
