"""Torch restatement of the per-face texture cubes mode (textures [B, nf, ts, ts, ts, 3], NR_FACE_TEXTURES): the
definition the fused kernels are checked against.  The reference has no renderer for these textures (DESIGN.md
"API notes"), so this is built from the oracle's own stages (oracle/pipeline.py) with the texture sampling swapped:
everything else -- z-buffer, weight map, lights, backgrounds, silhouettes, depth, flip, anti-aliasing and the
Differentiation stencil -- is the oracle's.  Gradients are what autograd gives through it."""
import itertools

import numpy as np
import torch

import oracle
from oracle import pipeline as ref


def sample_face_textures(faces, textures, fim, wmap, eps):
    """faces [B,nf,3,3] (gathered corners), textures [B,nf,ts,ts,ts,3], fim [B,R,R], wmap [B,R,R,3] -> rgb [B,R,R,3].

    Axis k of a face's cube belongs to its corner k: t_k = (q_k (ts-1) / zz_k) depth with the regularised depth of
    sample_textures, clamped to [0, max(ts-1-eps, 0)], then trilinear over the 8 texels around t.  A tap with an
    index >= ts reads as zero."""
    B, nf, ts = textures.shape[:3]
    tex = textures.reshape(B, nf * ts ** 3, 3)
    z_map = ref.to_map(faces[:, :, :, 2], fim)                      # [B,R,R,3]
    zz = z_map + 1e-10
    depth = 1. / (wmap / zz + 1e-10).sum(-1)                        # as in sample_textures
    t = (wmap * (ts - 1) / zz) * depth[..., None]
    t = torch.clamp(t, 0, max(ts - 1 - eps, 0))
    i = torch.floor(t)
    f = t - i
    i = i.long()
    base = fim.long() * ts ** 3
    rgb = 0
    for c in itertools.product((0, 1), repeat=3):
        j = [i[..., k] + c[k] for k in range(3)]
        ok = (fim >= 0) & (j[0] < ts) & (j[1] < ts) & (j[2] < ts)
        idx = torch.where(ok, base + (j[0] * ts + j[1]) * ts + j[2], -1)
        w = ((f[..., 0] if c[0] else 1 - f[..., 0]) * (f[..., 1] if c[1] else 1 - f[..., 1]) *
             (f[..., 2] if c[2] else 1 - f[..., 2]))
        rgb = rgb + w[..., None] * ref.to_map(tex, idx)
    return ref.mask_foreground(rgb, fim)


def rasterize(vertices, faces, image_size, anti_aliasing, textures, near=0.1, far=100.0, eps=1e-5, draw_backside=True,
              draw_silhouettes=True, draw_depth=False, lights=None, backgrounds=None, return_maps=False):
    """oracle.pipeline.rasterize with draw_rgb and per-face texture cubes: vertices [B,nv,3] screen space, faces [nf,3]
    (shared by the views), textures [B,nf,ts,ts,ts,3] -> images [B,C,S,S]."""
    R = image_size * 2 if anti_aliasing else image_size
    fidx = torch.as_tensor(np.asarray(faces)).long()
    fv = vertices[:, fidx]
    fv_np = np.ascontiguousarray(fv.detach().cpu().numpy(), dtype=np.float32)
    fim = torch.from_numpy(oracle.face_index_map(fv_np, R, near, far, draw_backside))
    wmap = torch.from_numpy(oracle.weight_map(fv_np, fim.numpy()))
    coord = ref.compute_coordinate_map(fv, fim, wmap)
    rgb = sample_face_textures(fv, textures, fim, wmap, eps)
    if lights is not None:
        rgb = rgb * ref.light_color_weights(ref.compute_normal_map(vertices, fidx, fv, fim, wmap), lights)
    if backgrounds is not None:
        fg = (0 <= fim).to(torch.float32)[..., None]
        rgb = fg * rgb + (1 - fg) * torch.flip(backgrounds.permute(0, 2, 3, 1), dims=(1, 2))
    chans = [rgb]
    if draw_silhouettes:
        chans.append((0 <= fim).to(torch.float32)[..., None])
    if draw_depth:
        chans.append(ref.compute_depth_map(fv, fim, wmap)[..., None])
    images = torch.cat(chans, -1) if len(chans) > 1 else chans[0]
    images = ref.differentiation(images, coord)
    images = torch.flip(images.permute(0, 3, 1, 2), dims=(2, 3))
    if anti_aliasing:
        images = (images[:, :, 0::2, 0::2] + images[:, :, 1::2, 0::2] +
                  images[:, :, 0::2, 1::2] + images[:, :, 1::2, 1::2]) / 4.
    if return_maps:
        return images, dict(face_index_map=fim, weight_map=wmap)
    return images
