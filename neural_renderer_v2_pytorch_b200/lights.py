"""Light sources, same classes and constructor arguments as the reference
(``neural_renderer_torch/lights.py:4-39``).  ``color`` / ``direction`` are [B,3] tensors (one row per
view), ``alpha`` is [B].  Shading itself runs inside the fused raster / backward kernels
(``csrc/nr_common.cuh::light_weights``, reference ``rasterize.py:252-283``).

The lights are differentiable like in the reference (where they flow through torch ops, rasterize.py:256-283):
a ``color`` / ``direction`` / ``alpha`` that requires grad receives its gradient from the fused backward
(``nr_rasterize_backward_lights``), through the packed [L,B,8] light data built here with torch ops.  A light
shared by all views is passed as ``param.expand(B, 3)``; autograd then sums its gradient over the views.  The
direction of a specular light is the fixed eye vector (0, 0, 1) and has no gradient."""
import torch


class Light:
    def __init__(self, color):
        self.color = color

    def to(self, device):
        self.color = self.color.to(device)


class DirectionalLight(Light):
    def __init__(self, color, direction, backside=False):
        super().__init__(color)
        self.direction = direction
        self.backside = backside

    def to(self, device):
        super().to(device)
        self.direction = self.direction.to(device)


class AmbientLight(Light):
    def __init__(self, color):
        super().__init__(color)


class SpecularLight(Light):
    def __init__(self, color, alpha=None, backside=False):
        super().__init__(color)
        self.backside = backside
        self.alpha = alpha if alpha is not None else torch.ones(color.shape[0], dtype=torch.float32)

    def to(self, device):
        super().to(device)
        self.alpha = self.alpha.to(device)


# (light types, device) -> int32 tensor of the types: made once, so a step captured in a CUDA graph copies nothing
# from the host for it
_types_cache = {}


def _f32(x, device):
    """Light parameter -> float32 tensor on ``device``, differentiable when ``x`` is a tensor that requires grad."""
    if torch.is_tensor(x):
        return x.to(device=device, dtype=torch.float32)
    return torch.as_tensor(x, dtype=torch.float32).to(device)


def pack_lights(lights, batch, device):
    """-> (types [L] int32, data [L,B,8] float32) on ``device``.

    ``data[l, b]`` = colour rgb, direction xyz, alpha, unused (include/nr_b200.h: nrLights).  It is built with torch
    ops, so light tensors that require grad stay connected to it: the fused backward returns d loss / d data and
    autograd routes it to each light's ``color`` / ``direction`` / ``alpha``."""
    types, rows = [], []
    device = torch.device(device)
    if len(lights) == 0:
        # `lights=[]` is "lit by nothing": a black image in the reference (the accumulated colour weight stays 0)
        lights = [AmbientLight(torch.zeros((batch, 3), dtype=torch.float32, device=device))]
    for light in lights:
        color = _f32(light.color, device)
        assert color.shape == (batch, 3), "light colour must be [batch, 3]"
        direction = alpha = None
        if isinstance(light, AmbientLight):
            t = 0
        elif isinstance(light, DirectionalLight):
            t = 1 | (4 if light.backside else 0)
            direction = _f32(light.direction, device)
        elif isinstance(light, SpecularLight):
            t = 2 | (4 if light.backside else 0)
            alpha = _f32(light.alpha, device)
        else:
            raise TypeError("unknown light type %r" % type(light))
        zeros = torch.zeros((batch, 8), dtype=torch.float32, device=device)
        row = torch.cat([color.expand(batch, 3),
                         direction.expand(batch, 3) if direction is not None else zeros[:, 3:6],
                         alpha.expand(batch)[:, None] if alpha is not None else zeros[:, 6:7],
                         zeros[:, 7:8]], dim=1)
        types.append(t)
        rows.append(row)
    key = (tuple(types), device)
    types_t = _types_cache.get(key)
    if types_t is None:
        types_t = _types_cache[key] = torch.tensor(types, dtype=torch.int32, device=device)
    return types_t, torch.stack(rows, 0).contiguous()


def vertex_normals(vertices, faces, deterministic=False):
    """Normalised per-vertex normals [B,nv,3] (``rasterize.py:167-182``): the cross products
    (v1-v0) x (v2-v1) of the faces touching a vertex, each face counted once per vertex, summed with
    index_add instead of the reference's dense [nf,nv] incidence matrix.  Differentiable torch ops.

    index_add sums with float atomics on CUDA, so the last bits vary from run to run.  ``deterministic`` sums
    with index_put(accumulate=True) instead, which sorts the indices and adds in a fixed order: the normals,
    and through them the lit images and every lit gradient, are then bit-identical from run to run.

    ``faces`` may also be [B,nf,3], one topology per view: view b's normals then come from row b alone, equal to
    a call with that view and row (the sums run over the flattened [B*nv] vertices, each view at its offset)."""
    import torch.nn.functional as F
    idx = faces.long()
    if idx.ndim == 3:
        B, nv = vertices.shape[:2]
        fv = vertices[torch.arange(B, device=idx.device)[:, None, None], idx]       # [B,nf,3,3]
        n = torch.linalg.cross(fv[:, :, 1] - fv[:, :, 0], fv[:, :, 2] - fv[:, :, 1], dim=-1)
        once1 = (idx[:, :, 1] != idx[:, :, 0]).to(n.dtype)[..., None]
        once2 = ((idx[:, :, 2] != idx[:, :, 0]) & (idx[:, :, 2] != idx[:, :, 1])).to(n.dtype)[..., None]
        flat = idx + (torch.arange(B, device=idx.device) * nv)[:, None, None]   # ids into [B*nv]
        vflat = vertices.reshape(B * nv, 3)
        if deterministic:
            # per view the same order of contributions as the [nf,3] call: corner 0 of every face, then 1, then 2
            vals = torch.cat([n, n * once1, n * once2], dim=1).reshape(-1, 3)
            ids = torch.cat([flat[:, :, 0], flat[:, :, 1], flat[:, :, 2]], dim=1).reshape(-1)
            vn = torch.zeros_like(vflat).index_put((ids,), vals, accumulate=True)
        else:
            vn = torch.zeros_like(vflat)
            vn = vn.index_add(0, flat[:, :, 0].reshape(-1), n.reshape(-1, 3))
            vn = vn.index_add(0, flat[:, :, 1].reshape(-1), (n * once1).reshape(-1, 3))
            vn = vn.index_add(0, flat[:, :, 2].reshape(-1), (n * once2).reshape(-1, 3))
        return F.normalize(vn.reshape(B, nv, 3), dim=2)
    fv = vertices[:, idx]                                            # [B,nf,3,3]
    n = torch.linalg.cross(fv[:, :, 1] - fv[:, :, 0], fv[:, :, 2] - fv[:, :, 1], dim=-1)
    once1 = (idx[:, 1] != idx[:, 0]).to(n.dtype)[None, :, None]
    once2 = ((idx[:, 2] != idx[:, 0]) & (idx[:, 2] != idx[:, 1])).to(n.dtype)[None, :, None]
    if deterministic:
        vals = torch.cat([n, n * once1, n * once2], dim=1).transpose(0, 1)     # [3nf,B,3]
        ids = torch.cat([idx[:, 0], idx[:, 1], idx[:, 2]])
        vn = torch.zeros_like(vertices.transpose(0, 1)).index_put((ids,), vals, accumulate=True).transpose(0, 1)
        return F.normalize(vn, dim=2)
    vn = torch.zeros_like(vertices)
    vn = vn.index_add(1, idx[:, 0], n)
    vn = vn.index_add(1, idx[:, 1], n * once1)
    vn = vn.index_add(1, idx[:, 2], n * once2)
    return F.normalize(vn, dim=2)
