"""``Mesh`` (reference ``neural_renderer_torch/mesh.py:8-37``): an ``nn.Module`` holding the vertices
of an .obj file and a learnable legacy (v1, 6-D) texture tensor: one ``ts^3`` RGB cube per face.

The reference leaves it half-ported (SURVEY.md section 2, row 11): nothing there renders its textures.
Here the three tensors of ``get_batch(B)`` render and differentiate as they are: faces ``[B, nf, 3]`` are
per-view meshes, and textures ``[B, nf, ts, ts, ts, 3]`` with ``None`` for both uv inputs select the
per-face texture cubes of the fused kernels (DESIGN.md "API notes"), e.g.
``renderer.render(v, f, None, None, t)``.  Differences: ``faces`` is kept as a tensor (the reference calls
``.expand`` on a numpy array, mesh.py:31) and ``to()`` returns the module."""
import torch
import torch.nn as nn

from .load_obj import load_obj


class Mesh(nn.Module):
    def __init__(self, filename_obj, texture_size=4, normalization=True):
        super().__init__()
        geometry = load_obj(filename_obj, normalization)
        self.vertices, self.faces = (torch.as_tensor(x) for x in geometry)   # mesh.py:14: plain tensors, not Parameters
        self.num_vertices, self.num_faces = len(self.vertices), len(self.faces)
        self.texture_size = texture_size
        # legacy v1 texture cube per face, normal-initialised (mesh.py:19-20)
        self.textures = nn.Parameter(torch.randn(self.num_faces, *([texture_size] * 3), 3))

    def to(self, *args, **kwargs):
        super().to(*args, **kwargs)
        device = torch._C._nn._parse_to(*args, **kwargs)[0]
        if device is not None:
            self.faces = self.faces.to(device)
            self.vertices = self.vertices.to(device)
        return self

    def get_batch(self, batch_size):
        """Broadcast to a minibatch (mesh.py:28-33); textures go through a sigmoid."""
        def tile(t):
            return t.unsqueeze(0).expand(batch_size, *t.shape)
        return tile(self.vertices), tile(self.faces), torch.sigmoid(tile(self.textures))

    def set_lr(self, lr_vertices, lr_textures):
        """Per-tensor learning-rate factors read by :class:`Adam` (mesh.py:35-37)."""
        for tensor, factor in ((self.vertices, lr_vertices), (self.textures, lr_textures)):
            tensor.lr = factor
