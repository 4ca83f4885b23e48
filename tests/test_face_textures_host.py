"""Per-face texture cubes ([B, nf, ts, ts, ts, 3], NR_FACE_TEXTURES) without a GPU: the torch definition
(face_textures_oracle.sample_face_textures) against a direct transcription of the v1 renderer's trilinear sampling,
known answers, float64 central differences, and the host's shape checks."""
import itertools

import numpy as np
import pytest
import torch

import neural_renderer_v2_pytorch_b200 as nr
from face_textures_oracle import sample_face_textures


def _pixels(seed, B=2, nf=5, R=12, ts=4, dtype=torch.float32, zlo=1., zhi=10.):
    """Random foreground pixels: face index map, normalised weights, corner depths in [zlo, zhi], cubes."""
    g = torch.Generator().manual_seed(seed)
    fim = torch.randint(0, nf, (B, R, R), generator=g, dtype=torch.int32)
    fim[:, 0, :3] = -1                                      # a few background pixels
    w = torch.rand((B, R, R, 3), generator=g, dtype=torch.float64) + 1e-3
    wmap = (w / w.sum(-1, keepdim=True)).to(dtype)
    faces = torch.zeros((B, nf, 3, 3), dtype=dtype)
    faces[..., 2] = (zlo + (zhi - zlo) * torch.rand((B, nf, 3), generator=g, dtype=torch.float64)).to(dtype)
    tex = torch.rand((B, nf, ts, ts, ts, 3), generator=g, dtype=torch.float64).to(dtype)
    return faces, tex, fim, wmap


def _v1(faces, tex, fim, wmap, eps):
    """The v1 renderer's per-face texture lookup, in float64: unregularised depth 1 / sum(w / z), texel position
    w_k (ts - 1) depth / z_k clamped to [0, ts - 1 - eps], truncating (int), index i0 ts^2 + i1 ts + i2."""
    faces, tex, fim, wmap = (np.asarray(x, np.float64) if x.dtype.is_floating_point else np.asarray(x)
                             for x in (faces, tex, fim, wmap))
    B, nf, ts = tex.shape[:3]
    out = np.zeros(fim.shape + (3,))
    for b, y, x in zip(*np.nonzero(fim >= 0)):
        f = fim[b, y, x]
        w, z = wmap[b, y, x], faces[b, f, :, 2]
        depth = 1. / np.sum(w / z)
        pos = np.clip(w * (ts - 1) * depth / z, 0, ts - 1 - eps)
        pi = pos.astype(np.int64)
        pf = pos - pi
        cube = tex[b, f].reshape(ts ** 3, 3)
        for c in itertools.product((0, 1), repeat=3):
            wt = np.prod([pf[k] if c[k] else 1 - pf[k] for k in range(3)])
            out[b, y, x] += wt * cube[(pi[0] + c[0]) * ts * ts + (pi[1] + c[1]) * ts + pi[2] + c[2]]
    return out


@pytest.mark.parametrize("ts", [2, 3, 4, 7])
def test_matches_the_v1_formula(ts):
    faces, tex, fim, wmap = _pixels(ts, ts=ts)
    got = sample_face_textures(faces, tex, fim, wmap, 1e-5).numpy()
    want = _v1(faces, tex, fim, wmap, 1e-5)
    assert np.abs(got - want).max() <= 1e-6, np.abs(got - want).max()
    assert np.abs(want).max() > 0.1


@pytest.mark.parametrize("ts", [2, 4, 5])
def test_affine_cube_is_reproduced_exactly(ts):
    """Trilinear interpolation reproduces affine data: the sample of a cube holding a + b . (i0, i1, i2) is a + b . t."""
    faces, _, fim, wmap = _pixels(10 + ts, ts=ts, dtype=torch.float64)
    B, nf = faces.shape[:2]
    a = torch.tensor([0.25, -1.0, 3.0], dtype=torch.float64)
    bk = torch.tensor([[0.5, -0.25, 2.0], [1.5, 0.75, -0.5], [-2.0, 0.125, 1.0]], dtype=torch.float64)   # [axis, rgb]
    i = torch.stack(torch.meshgrid(*[torch.arange(ts, dtype=torch.float64)] * 3, indexing="ij"), -1)   # [ts,ts,ts,3]
    cube = a + i @ bk
    tex = cube.expand(B, nf, ts, ts, ts, 3).contiguous()
    got = sample_face_textures(faces, tex, fim, wmap, 1e-5)
    # t from the definition, independently
    z = faces[..., 2][torch.arange(B)[:, None, None], fim.clamp(min=0).long()]
    zz = z + 1e-10
    depth = 1. / (wmap / zz + 1e-10).sum(-1, keepdim=True)
    t = (wmap * (ts - 1) / zz * depth).clamp(0, ts - 1 - 1e-5)
    want = torch.where((fim >= 0)[..., None], a + t @ bk, torch.zeros((), dtype=torch.float64))
    assert torch.allclose(got, want, rtol=0, atol=1e-12), (got - want).abs().max()


def test_one_texel_per_face():
    """ts = 1: every pixel of a face shows its one texel."""
    faces, tex, fim, wmap = _pixels(3, ts=1)
    got = sample_face_textures(faces, tex, fim, wmap, 1e-5)
    B = fim.shape[0]
    want = tex.reshape(B, -1, 3)[torch.arange(B)[:, None, None], fim.clamp(min=0).long()]
    want = torch.where((fim >= 0)[..., None], want, torch.zeros(()))
    assert torch.equal(got, want)


def test_gradients_match_central_differences():
    """Autograd of the definition against float64 central differences, for the textures and the corner depths, at
    pixels away from cell boundaries and from the clamp (where t is not differentiable)."""
    ts, eps = 4, 1e-5
    faces, tex, fim, wmap = _pixels(7, B=1, nf=3, R=6, ts=ts, dtype=torch.float64, zlo=1., zhi=3.)
    with torch.no_grad():
        z = faces[..., 2][torch.arange(1)[:, None, None], fim.clamp(min=0).long()]
        depth = 1. / (wmap / (z + 1e-10) + 1e-10).sum(-1, keepdim=True)
        t = wmap * (ts - 1) / (z + 1e-10) * depth
        fr = t - torch.floor(t)
        smooth = ((fr > 0.02) & (fr < 0.98) & (t > 0) & (t < ts - 1 - eps)).all(-1) & (fim >= 0)
    assert smooth.sum() >= 8, "too few smooth pixels"
    fim = torch.where(smooth, fim, torch.full_like(fim, -1))
    G = torch.randn(fim.shape + (3,), generator=torch.Generator().manual_seed(1), dtype=torch.float64)

    def loss(texv, zv):
        fv = faces.clone()
        fv[..., 2] = zv
        return (sample_face_textures(fv, texv, fim, wmap, eps) * G).sum()

    assert torch.autograd.gradcheck(loss, (tex.clone().requires_grad_(True), faces[..., 2].clone().requires_grad_(True)),
                                    eps=1e-7, atol=1e-8, rtol=1e-6)


def _hp():
    return nr.RasterizeHyperparam(image_size=16, anti_aliasing=False)


@pytest.mark.parametrize("case", ["uv_given", "faces_textures_given", "wrong_nf", "wrong_batch", "not_a_cube",
                                  "channels_first"])
def test_bad_face_texture_shapes_raise_assertion_error(case):
    B, nf, ts = 3, 4, 2
    v = torch.zeros(B, 5, 3)
    f = torch.zeros(nf, 3, dtype=torch.int32)
    tex = torch.zeros(B, nf, ts, ts, ts, 3)
    vt = ft = None
    if case == "uv_given":
        vt = torch.zeros(B, 3, 2)
    elif case == "faces_textures_given":
        ft = torch.zeros(nf, 3, dtype=torch.int32)
    elif case == "wrong_nf":
        tex = torch.zeros(B, nf + 1, ts, ts, ts, 3)
    elif case == "wrong_batch":
        tex = torch.zeros(B - 1, nf, ts, ts, ts, 3)
    elif case == "not_a_cube":
        tex = torch.zeros(B, nf, ts, ts, ts + 1, 3)
    else:
        tex = torch.zeros(B, nf, 3, ts, ts, ts)
    p = nr.RasterizeParam(vertices_textures=vt, faces_textures=ft, textures=tex)
    with pytest.raises(AssertionError):
        nr.rasterize_rgb(v, f, p, _hp())


def test_per_view_faces_and_cubes_shape_check():
    """[B, nf, 3] faces with [B, nf, ts, ts, ts, 3] cubes pass the shape checks (and stop at the device check)."""
    B, nf, ts = 2, 4, 3
    p = nr.RasterizeParam(textures=torch.zeros(B, nf, ts, ts, ts, 3))
    with pytest.raises(RuntimeError, match="CUDA"):
        nr.rasterize_rgba(torch.zeros(B, 5, 3), torch.zeros(B, nf, 3, dtype=torch.int32), p, _hp())
    with pytest.raises(AssertionError):
        nr.rasterize_rgba(torch.zeros(B, 5, 3), torch.zeros(B, nf - 1, 3, dtype=torch.int32), p, _hp())
