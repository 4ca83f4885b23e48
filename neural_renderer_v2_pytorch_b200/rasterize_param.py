"""Parameter holders of the rasterize API, field-for-field the reference's
``neural_renderer_torch/rasterize_param.py:13-50`` (same names, same defaults)."""


class RasterizeHyperparam:
    def __init__(self, image_size=256, near=0.1, far=100.0, eps=1e-5, anti_aliasing=True,
                 draw_backside=True, draw_rgb=True, draw_silhouettes=True, draw_depth=True):
        self.image_size = image_size
        self.near = near
        self.far = far
        self.eps = eps
        self.anti_aliasing = anti_aliasing
        self.draw_backside = draw_backside
        self.draw_rgb = draw_rgb
        self.draw_silhouettes = draw_silhouettes
        self.draw_depth = draw_depth
        # not in the reference: bit-reproducible gradients (fixed-point sums in a unit chosen per view from its
        # max |grad_images|: exact under power-of-two loss scaling, NaN / inf as in float mode; see nr_b200.h)
        self.deterministic = False


class RasterizeParam:
    def __init__(self, vertices_textures=None, faces_textures=None, textures=None,
                 background_color=None, backgrounds=None, lights=None):
        self.vertices_textures = vertices_textures
        self.faces_textures = faces_textures
        self.textures = textures
        self.background_color = background_color
        self.backgrounds = backgrounds
        self.lights = lights
