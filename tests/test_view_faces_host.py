"""Host side of per-view faces ([B, nf, 3]): vertex normals and the shape checks (no GPU needed)."""
import pytest
import torch

import neural_renderer_v2_pytorch_b200 as nr
from neural_renderer_v2_pytorch_b200 import lights as light_lib


def _batch(seed=0, B=3, nv=7, nf=9):
    g = torch.Generator().manual_seed(seed)
    v = torch.randn(B, nv, 3, generator=g)
    f = torch.randint(0, nv, (B, nf, 3), generator=g)
    f[0, 0] = torch.tensor([2, 2, 5])            # a face that lists a vertex twice
    f[1, 3] = torch.tensor([4, 1, 4])
    f[2, 5] = torch.tensor([0, 0, 0])            # a padded (degenerate) face
    return v, f


@pytest.mark.parametrize("deterministic", [False, True])
def test_vertex_normals_per_view_equal_single_view_calls(deterministic):
    v, f = _batch()
    got = light_lib.vertex_normals(v, f, deterministic=deterministic)
    assert got.shape == v.shape
    for b in range(v.shape[0]):
        want = light_lib.vertex_normals(v[b:b + 1], f[b], deterministic=deterministic)
        assert torch.equal(got[b:b + 1], want), b


@pytest.mark.parametrize("deterministic", [False, True])
def test_vertex_normals_per_view_gradient_equals_single_view_calls(deterministic):
    v, f = _batch(seed=1)
    w = torch.randn(v.shape, generator=torch.Generator().manual_seed(2))
    v1 = v.clone().requires_grad_(True)
    (light_lib.vertex_normals(v1, f, deterministic=deterministic) * w).sum().backward()
    for b in range(v.shape[0]):
        v0 = v[b:b + 1].clone().requires_grad_(True)
        (light_lib.vertex_normals(v0, f[b], deterministic=deterministic) * w[b:b + 1]).sum().backward()
        assert torch.allclose(v1.grad[b:b + 1], v0.grad, rtol=1e-5, atol=1e-6), b


def test_vertex_normals_shared_faces_expanded_equal_shared_call():
    v, f = _batch(seed=3)
    shared = f[0]
    for det in (False, True):
        a = light_lib.vertex_normals(v, shared, deterministic=det)
        b = light_lib.vertex_normals(v, shared.expand(v.shape[0], *shared.shape), deterministic=det)
        assert torch.equal(a, b)


@pytest.mark.parametrize("faces_shape", [(2, 4, 3), (3, 4, 4), (3, 1, 4, 3)],
                         ids=["other_batch", "four_columns", "four_dims"])
def test_bad_faces_shapes_raise_assertion_error(faces_shape):
    hp = nr.RasterizeHyperparam(image_size=16, anti_aliasing=False)
    v = torch.zeros(3, 5, 3)
    f = torch.zeros(faces_shape, dtype=torch.int32)
    with pytest.raises(AssertionError):
        nr.rasterize_silhouettes(v, f, nr.RasterizeParam(), hp)
