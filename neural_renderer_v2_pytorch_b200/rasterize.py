"""Host side of the rasterize path: same public functions as the reference's
``neural_renderer_torch/rasterize.py`` (``rasterize_silhouettes`` :332-338, ``rasterize_rgba``
:341-347, ``rasterize_rgb`` :350-356, ``rasterize_depth`` :359-365, ``rasterize_core`` :194-329),
driving ONE fused CUDA forward and ONE fused CUDA backward through the C ABI instead of ~60
torch ops with per-view host synchronisation.

Differences from the reference that are deliberate (DESIGN.md "API notes"):
  * ``hyperparams.image_size`` is NOT doubled in place when anti-aliasing is on
    (the reference mutates the caller's object, rasterize.py:227-228);
  * ``backgrounds`` / ``background_color`` work: the reference's ``blend_backgrounds``
    (rasterize.py:156-159) fails on torch tensors (``.astype`` / ``[::-1]``) and its ``background_color``
    multiplies a zero tensor (:208-215); here they do what the Chainer original blends
    (neural_renderer_chainer/rasterize.py:574-577) with a constant colour that is actually the colour.
"""
import ctypes
import os

import torch

from . import _lib
from . import lights as light_lib
from .rasterize_param import RasterizeParam, RasterizeHyperparam

DEPTH_MIN_DELTA = 1e-4      # rasterize.py:35

# Deterministic backward (bit-identical gradients from run to run): set to True, or per call through
# RasterizeHyperparam(...).deterministic = True.  Costs one int64 scratch buffer per backward.
DETERMINISTIC = False

# test hook: bin into 8x8 tiles (dense-mesh mode of the general path) whatever the statistics say
FORCE_FINE_TILES = False

# Tile lists longer than this (nrBinStats.max_tile_faces of an earlier call) switch a shape that is binned
# by the general path to 8x8 tiles.
FINE_TILES_ABOVE = 192

# test hook: True / False forces the face-parallel raster kernel for meshes of small triangles (nr_raster_dense.cu)
# on / off whatever the statistics say; None = decide from the statistics of earlier calls
FORCE_DENSE_RASTER = {"0": False, "1": True}.get(os.environ.get("NR_FORCE_DENSE_RASTER", ""))

# A shape binned by the general path whose tile lists hold this many faces on average (nrBinStats.total_pairs over
# the tiles of the batch, from an earlier call) is rasterized by the face-parallel kernel.
DENSE_RASTER_ABOVE = 32

# Forward -> backward state (nr_b200.h: aux_map): the forward stores the normalised weights and the texel
# coordinate of every foreground pixel, the backward reads them instead of re-deriving them (9 scattered vertex
# loads and 12 IEEE divisions per pixel).  Measured at config 2 (profiles/r2_aux_map_ab.txt): the backward gets
# 4 us faster, the forward 5 us slower (100 MB more to write) - a wash, so it is off unless asked for.
USE_AUX_MAP = os.environ.get("NR_USE_AUX_MAP", "0") == "1"

# test hook: always bin with the general multi-kernel path (large meshes) instead of the one-kernel path
FORCE_GENERAL_BINNING = False

# test hook: force the (tile, face) pair capacity (e.g. 0) to exercise the device-side overflow path
FORCE_PAIR_CAPACITY = None


def _require_cuda(t, name):
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if not t.is_cuda:
        # same error class and wording as CHECK_CUDA, rasterize_cuda.cpp:5
        raise RuntimeError("%s must be a CUDA tensor" % name)


def _f32c(t):
    return t.detach().to(torch.float32).contiguous()


def _i32c(t):
    return t.detach().to(torch.int32).contiguous()


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class _Scratch:
    """Per (device, stream) scratch: workspace bytes, pinned bin statistics, a CUDA event.

    The forward never waits for the GPU.  The bin statistics of call k are read when call k+1
    (or later) finds their event complete; if the (tile, face) pair list overflowed, call k was
    still correct (device-side fallback, see nr_b200.h) and the capacity grows for the next call."""

    _cache = {}

    def __init__(self, device):
        self.device = device
        self.workspace = None
        self.pair_capacity = 0
        self.stats = torch.zeros(4, dtype=torch.int32).pin_memory()
        self.pending = False
        self.overflows = 0
        self.general_binning = set()        # (nf, R) whose views outgrew the one-kernel small-mesh binning
        self.fine_tiles = set()             # (nf, R) dense enough for 8x8 tiles (general path only)
        self.dense = set()                  # (nf, R) of small triangles: face-parallel z-buffer rasterizer
        self.not_dense = set()              # ... that turned out to hold too many large faces for it
        self.last_dense = False
        self.last_tiles = 1
        self.last_faces = 0
        self.bad_index = 0                  # nrBinStats.bad_index bits seen and not yet reported
        self.last_shape = None
        self.last_small = True
        ev = ctypes.c_void_p()
        _lib.check(_lib.lib().nr_event_create(ctypes.byref(ev)), "nr_event_create")
        self.event = ev

    @classmethod
    def get(cls, device, stream):
        key = (device.index, stream)
        s = cls._cache.get(key)
        if s is None:
            s = cls._cache[key] = cls(device)
        return s

    def poll(self, block=False):
        """Fold the statistics of the last launched forward into the capacity, if they have arrived."""
        if not self.pending:
            return
        L = _lib.lib()
        if block:
            _lib.check(L.nr_event_synchronize(self.event), "nr_event_synchronize")
        elif L.nr_event_query(self.event) != 1:
            return
        self.pending = False
        total, max_tile, overflow, bad = self.stats.tolist()
        if self.last_dense:
            # z-buffer path: total = contested pixels, max_tile = faces with a pixel box above 4096 pixels
            if max_tile * 50 > self.last_faces and self.last_shape is not None:
                self.dense.discard(self.last_shape)
                self.not_dense.add(self.last_shape)
        elif self.last_shape is not None and not self.last_small:
            if max_tile > FINE_TILES_ABOVE:
                self.fine_tiles.add(self.last_shape)
            # many faces per tile, few tiles per face: small triangles
            if (total >= DENSE_RASTER_ABOVE * self.last_tiles and total <= 3 * self.last_faces
                    and self.last_shape not in self.not_dense):
                self.dense.add(self.last_shape)
        self.bad_index |= bad
        if overflow:
            self.overflows += 1
            if self.last_dense:
                self.pair_capacity = min(max(self.pair_capacity * 4, 1 << 20), 0x7fffffff)
            else:
                self.pair_capacity = max(self.pair_capacity, int(total * 1.25) + 4096)
            if overflow == 2:
                self.general_binning.add(self.last_shape)

    def report_bad_indices(self):
        """An earlier call on this stream dropped faces (bit 0) or drew black pixels (bit 1) because of an index
        outside its range: the reference raises IndexError for those (rasterize.py:232,246).  The synchronous
        check (_validate_indices) catches them first on every eager call; this one covers calls replayed from a
        CUDA graph, whose index tensors were edited after the capture."""
        bad, self.bad_index = self.bad_index, 0
        if bad:
            what = " and ".join(n for bit, n in ((1, "faces (vertex index)"), (2, "faces_textures (texture-vertex index)")) if bad & bit)
            raise IndexError("an earlier rasterize call on this stream had out-of-range indices in %s; "
                             "those faces were dropped / drawn black" % what)

    def ensure(self, cfg, capacity):
        need = _lib.lib().nr_workspace_bytes(ctypes.byref(cfg), capacity)
        if self.workspace is None or self.workspace.numel() < need:
            # torch's caching allocator hands out 512-byte aligned blocks.  (A workspace a captured CUDA graph
            # replays on stays alive through the reference its replay object holds, see graph.capture_step.)
            self.workspace = torch.empty(int(need * 1.25) + 256, dtype=torch.uint8, device=self.device)
        self.pair_capacity = capacity


# graph.capture_step sets this to a list while it captures: every workspace a captured forward bakes into the
# graph is appended, and the replay object keeps the list, so a later, larger problem on the same stream cannot
# free memory a graph still replays on
_capture_keepalive = None


def _make_config(B, nv, nf, S, flags, hp, nvt=0, H=0, W=0):
    return _lib.RasterConfig(batch=B, num_vertices=nv, num_faces=nf, image_size=S, flags=flags,
                             near_plane=float(hp.near), far_plane=float(hp.far), eps=float(hp.eps),
                             depth_min_delta=DEPTH_MIN_DELTA, num_tex_vertices=nvt, tex_height=H,
                             tex_width=W)


def _flags_of(hp):
    return ((_lib.NR_DRAW_RGB if hp.draw_rgb else 0) |
            (_lib.NR_DRAW_SILHOUETTES if hp.draw_silhouettes else 0) |
            (_lib.NR_DRAW_DEPTH if hp.draw_depth else 0) |
            (_lib.NR_DRAW_BACKSIDE if hp.draw_backside else 0) |
            (_lib.NR_ANTI_ALIASING if hp.anti_aliasing else 0) |
            (_lib.NR_DETERMINISTIC if (DETERMINISTIC or getattr(hp, "deterministic", False)) else 0))


def _lights_struct(lights, grad_vn=None, backgrounds=None):
    """lights = (types, data, vertex_normals) or None, backgrounds [B,3,R,R] or None
    -> ctypes nrLights pointer or None."""
    if lights is None and backgrounds is None:
        return None
    bg = backgrounds.data_ptr() if backgrounds is not None else None
    if lights is None:
        return ctypes.byref(_lib.Lights(num_lights=0, backgrounds=bg))
    types, data, vn = lights
    return ctypes.byref(_lib.Lights(num_lights=types.shape[0], types=types.data_ptr(), data=data.data_ptr(),
                                    vertex_normals=vn.data_ptr(),
                                    grad_vertex_normals=grad_vn.data_ptr() if grad_vn is not None else None,
                                    backgrounds=bg))


def _zero_fill_struct(buffers):
    """Tensors the forward zero-fills on the side (see nrZeroFill) -> ctypes pointer or None."""
    buffers = [t for t in buffers if t is not None and t.numel()]
    if not buffers:
        return None
    z = _lib.ZeroFill(count=len(buffers))
    for i, t in enumerate(buffers):
        z.ptr[i] = t.data_ptr()
        z.bytes[i] = t.numel() * t.element_size()
    return ctypes.byref(z)


def _forward_call(cfg, vertices, faces, vt, ft, tex, want_maps, lights=None, backgrounds=None, zero=(), sparse=False,
                  want_aux=False):
    """Enqueues nr_rasterize_forward on the current stream and returns without synchronising.
    Returns (images, internal, fim, wmap, dmap, tile_list, aux)."""
    L = _lib.lib()
    dev = vertices.device
    B, S = cfg.batch, cfg.image_size
    aa = bool(cfg.flags & _lib.NR_ANTI_ALIASING)
    R = S * 2 if aa else S
    C = L.nr_num_channels(cfg.flags)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        sc = _Scratch.get(dev, stream)
        # inside a CUDA-graph capture nothing may query or synchronise: the statistics of the
        # eager warm-up calls have already sized the workspace
        capturing = torch.cuda.is_current_stream_capturing()
        if not capturing:
            sc.poll()
            sc.report_bad_indices()
        fim = torch.empty((B, R, R), dtype=torch.int32, device=dev)
        images = torch.empty((B, C, S, S), dtype=torch.float32, device=dev)
        internal = torch.empty((B, C, R, R), dtype=torch.float32, device=dev) if aa else None
        wmap = torch.empty((B, R, R, 3), dtype=torch.float32, device=dev) if want_maps else None
        dmap = torch.empty((B, R, R), dtype=torch.float32, device=dev) if want_maps else None
        # forward -> backward state (weights and texel coordinates of the foreground pixels, see nr_b200.h)
        aux = None
        if want_aux and not (cfg.flags & _lib.NR_DETERMINISTIC):
            aux = torch.empty((B, R, R, 6 if (cfg.flags & _lib.NR_DRAW_RGB) else 3), dtype=torch.float32, device=dev)
        # which binning this call takes: one kernel per view (small meshes), the general path, or the
        # general path over 8x8 tiles (dense meshes); the last two are learnt from earlier calls' statistics
        shape = (cfg.num_faces, R)
        general = shape in sc.general_binning or FORCE_GENERAL_BINNING
        small = cfg.num_faces <= 8192 and ((R + 15) // 16) ** 2 <= 4096 and not general
        dense = (not small and shape in sc.dense) if FORCE_DENSE_RASTER is None else bool(FORCE_DENSE_RASTER)
        fine = not dense and (FORCE_FINE_TILES or (not small and shape in sc.fine_tiles))
        if general:
            cfg.flags |= _lib.NR_GENERAL_BINNING
        if fine:
            cfg.flags |= _lib.NR_FINE_TILES
        if dense:
            cfg.flags |= _lib.NR_DENSE_RASTER
        tile = 8 if fine else 16
        ntx = (R + tile - 1) // tile
        tile_list = torch.empty(8 + 16 * B * ntx * ntx, dtype=torch.int32, device=dev)
        capacity = max(sc.pair_capacity, 4 * B * cfg.num_faces + 4096)
        if FORCE_PAIR_CAPACITY is not None:
            capacity = int(FORCE_PAIR_CAPACITY)
        need_grow = sc.workspace is None or sc.workspace.numel() < L.nr_workspace_bytes(ctypes.byref(cfg), capacity)
        if capturing and need_grow:
            raise RuntimeError("run the step eagerly a few times before capturing it in a CUDA graph "
                               "(the rasterizer sizes its workspace from those warm-up calls)")
        if sc.pending and not capturing:
            # the pinned statistics are still owned by an earlier call in flight
            sc.poll(block=need_grow)
        sc.ensure(cfg, capacity)
        ws = sc.workspace
        base = ws.data_ptr()
        aligned = (base + 255) & ~255
        track = not sc.pending and not capturing
        if sparse and not want_maps and not fine:
            cfg.flags |= _lib.NR_SPARSE_MAPS     # fim / internal image are only handed to the backward
        if track:
            sc.last_shape, sc.last_small, sc.last_tiles = shape, small, B * ((R + 15) // 16) ** 2
            sc.last_dense, sc.last_faces = dense, B * cfg.num_faces
        if capturing and _capture_keepalive is not None:
            _capture_keepalive.append(ws)
        rc = L.nr_rasterize_forward(
            ctypes.byref(cfg), _ptr(vertices), _ptr(faces), _ptr(vt), _ptr(ft), _ptr(tex),
            _ptr(fim), _ptr(wmap), _ptr(dmap), _ptr(images), _ptr(internal), _ptr(aux), _ptr(tile_list),
            ctypes.c_void_p(aligned), ws.numel() - (aligned - base), capacity,
            ctypes.c_void_p(sc.stats.data_ptr()) if track else None, sc.event if track else None,
            _zero_fill_struct(zero), _lights_struct(lights, None, backgrounds), ctypes.c_void_p(stream))
        _lib.check(rc, "nr_rasterize_forward")
        if track:
            sc.pending = True
        # with 8x8 tiles the list is of no use to the backward (it walks 16x16 tiles)
        return images, internal, fim, wmap, dmap, (None if fine else tile_list), aux


def _validate_indices(idx, limit, what):
    """Index range check with the reference's error type (IndexError from tensor indexing,
    rasterize.py:232,246).  Costs one device->host read per index TENSOR and version of its contents: the
    verdict is remembered on the tensor object itself (it dies with it, so a new tensor at a recycled address
    is checked again).  Safety does not rest on this check: the kernels test every index themselves
    (nrBinStats.bad_index, reported by the next call on the stream)."""
    key = (idx._version, limit)
    if getattr(idx, "_nr_validated", None) == key:
        return
    if idx.is_cuda and torch.cuda.is_current_stream_capturing():
        return      # cannot read back during capture; the kernels drop out-of-range faces anyway
    if idx.numel():
        lo, hi = int(idx.min()), int(idx.max())
        if lo < 0 or hi >= limit:
            raise IndexError("%s reference index %d outside [0, %d)" % (what, hi if hi >= limit else lo, limit))
    if idx.is_cuda:         # a CPU tensor may share memory with a numpy array edited behind torch's back
        try:
            idx._nr_validated = key
        except (AttributeError, RuntimeError):
            pass


class _Rasterize(torch.autograd.Function):
    """Forward: nr_rasterize_forward. Backward: nr_rasterize_backward_lights (Differentiation stencil +
    every autograd edge the reference has on this path, the light parameters included).  ``light_data`` is the
    [L,B,8] tensor of lights.pack_lights, an input of its own so that autograd sees it; ``light_types`` its [L]
    types."""

    @staticmethod
    def forward(ctx, vertices, vertices_textures, textures, vertex_normals, backgrounds, light_data, faces,
                faces_textures, cfg, light_types):
        v = _f32c(vertices)
        bg = _f32c(backgrounds) if backgrounds is not None else None
        vt = _f32c(vertices_textures) if vertices_textures is not None else None
        tex = _f32c(textures) if textures is not None else None
        lights = None
        if light_data is not None:
            lights = (light_types, _f32c(light_data), _f32c(vertex_normals))
        # The backward ADDS into its outputs.  When a backward is coming its accumulators are allocated
        # here and zero-filled by the raster kernel on the side (nrZeroFill) instead of by separate
        # fill kernels in front of the backward.
        need = ctx.needs_input_grad
        ctx.grad_bufs = None
        if any(need[:3]):
            gv = torch.empty_like(v) if need[0] else None
            gvt = torch.empty_like(vt) if (need[1] and vt is not None) else None
            gtex = torch.empty_like(tex) if (need[2] and tex is not None) else None
            if gv is not None or gvt is not None or gtex is not None:
                ctx.grad_bufs = (gv, gvt, gtex)
        images, internal, fim, _, _, tile_list, aux = _forward_call(cfg, v, faces, vt, faces_textures, tex, False, lights, bg,
                                                                    ctx.grad_bufs or (),
                                                                    sparse=not (bg is not None and need[4]),
                                                                    want_aux=USE_AUX_MAP and ctx.grad_bufs is not None)
        ctx.cfg = cfg
        ctx.bg_dtype = backgrounds.dtype if backgrounds is not None else None
        ctx.has_tex = tex is not None
        ctx.has_lights = lights is not None
        ctx.in_dtypes = tuple(t.dtype if t is not None else None
                              for t in (vertices, vertices_textures, textures, vertex_normals, light_data))
        ctx.has_aux = aux is not None
        saved = [v, faces, fim, internal if internal is not None else images, tile_list]
        if ctx.has_aux:
            saved.append(aux)
        if ctx.has_tex:
            saved += [vt, faces_textures, tex]
        if ctx.has_lights:
            saved += list(lights)
        ctx.save_for_backward(*saved)
        return images

    @staticmethod
    def backward(ctx, grad_images):
        cfg = ctx.cfg
        L = _lib.lib()
        saved = list(ctx.saved_tensors)
        lights = tuple(saved[-3:]) if ctx.has_lights else None
        if ctx.has_lights:
            saved = saved[:-3]
        aux = saved.pop(5) if ctx.has_aux else None
        if ctx.has_tex:
            v, faces, fim, internal, tile_list, vt, ft, tex = saved
        else:
            v, faces, fim, internal, tile_list = saved
            vt = ft = tex = None
        g = _f32c(grad_images)
        need_v, need_vt, need_tex = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        gbg = None
        if ctx.bg_dtype is not None and ctx.needs_input_grad[4]:
            # blend backward: background pixels pass the rgb gradient straight to the picture
            # (output orientation = flipped internal orientation; 2x2 mean backward under AA)
            grgb = g[:, :3]
            if cfg.flags & _lib.NR_ANTI_ALIASING:
                grgb = (grgb * 0.25).repeat_interleave(2, dim=2).repeat_interleave(2, dim=3)
            gbg = (grgb * (torch.flip(fim, dims=(1, 2)) < 0)[:, None]).to(ctx.bg_dtype)
        dev = v.device
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            # accumulators zero-filled by the forward; a repeated backward (retain_graph) makes new ones
            pre, ctx.grad_bufs = (ctx.grad_bufs or (None, None, None)), None
            gv = pre[0] if pre[0] is not None else torch.zeros_like(v)
            gvt = (pre[1] if pre[1] is not None else torch.zeros_like(vt)) if (need_vt and vt is not None) else None
            gtex = (pre[2] if pre[2] is not None else torch.zeros_like(tex)) if (need_tex and tex is not None) else None
            gvn = torch.zeros_like(lights[2]) if (lights is not None and ctx.needs_input_grad[3]) else None
            # d loss / d light data [L,B,8] (colour, direction, alpha), summed by the backward kernel
            glight = torch.zeros_like(lights[1]) if (lights is not None and ctx.needs_input_grad[5]) else None
            scratch = lscratch = None
            if cfg.flags & _lib.NR_DETERMINISTIC:
                scratch = torch.zeros(L.nr_deterministic_scratch_bytes(ctypes.byref(cfg)) // 8, dtype=torch.int64, device=dev)
                if glight is not None:
                    lscratch = torch.zeros(glight.numel(), dtype=torch.int64, device=dev)
            rc = L.nr_rasterize_backward_lights(ctypes.byref(cfg), _ptr(v), _ptr(faces), _ptr(vt), _ptr(ft),
                                                _ptr(tex), _ptr(fim), _ptr(internal), _ptr(aux), _ptr(tile_list), _ptr(g),
                                                _ptr(gv), _ptr(gtex), _ptr(gvt), _ptr(scratch), _lights_struct(lights, gvn),
                                                _ptr(glight), _ptr(lscratch), ctypes.c_void_p(stream))
            _lib.check(rc, "nr_rasterize_backward_lights")
        cast = lambda g_, dt: g_.to(dt) if (g_ is not None and dt is not None and g_.dtype != dt) else g_
        dv, dvt, dtex, dvn, dlight = ctx.in_dtypes
        return ((cast(gv, dv) if need_v else None), cast(gvt, dvt), cast(gtex, dtex), cast(gvn, dvn), gbg,
                cast(glight, dlight), None, None, None, None)


def _prepare(vertices, faces, params, hyperparams):
    # shape checks of rasterize.py:195-205 (AssertionError, like the reference).  Beyond the reference, faces (and
    # faces_textures) may be [B, nf, 3]: one topology per view (NR_VIEW_FACES, DESIGN.md "API notes").
    assert vertices.ndim == 3
    assert vertices.shape[2] == 3
    assert faces.ndim in (2, 3)
    assert faces.shape[-1] == 3
    assert faces.ndim == 2 or faces.shape[0] == vertices.shape[0]
    dev = vertices.device
    bg = None
    if hyperparams.draw_rgb:
        # rasterize.py:207-225; backgrounds only ever touch the rgb channels (:286-288)
        R_ = int(hyperparams.image_size) * (2 if hyperparams.anti_aliasing else 1)
        if params.background_color is not None:
            color = torch.as_tensor(params.background_color, dtype=torch.float32, device=dev)
            assert color.shape == (3,)
            bg = color[None, :, None, None].expand(vertices.shape[0], 3, R_, R_)
        elif params.backgrounds is not None:
            bg = params.backgrounds
            assert bg.ndim == 4
            assert bg.shape[0] == vertices.shape[0]
            assert bg.shape[1] == 3
            assert bg.shape[2] == R_
            assert bg.shape[3] == R_
            _require_cuda(bg, "backgrounds")
    _require_cuda(vertices, "vertices")
    faces = torch.as_tensor(faces)
    faces_d = _i32c(faces).to(dev)
    B, nv = vertices.shape[:2]
    nf = faces_d.shape[-2]
    _validate_indices(faces, nv, "faces")
    view_faces = faces_d.ndim == 3
    vt = ft = tex = None
    nvt = H = W = 0
    if hyperparams.draw_rgb:
        assert params.vertices_textures.ndim == 3
        assert params.vertices_textures.shape[2] == 2
        assert params.faces_textures.ndim in (2, 3)
        assert params.faces_textures.shape[-1] == 3
        assert params.textures.ndim == 4
        assert params.textures.shape[1] == 3
        vt, tex = params.vertices_textures, params.textures
        _require_cuda(vt, "vertices_textures")
        _require_cuda(tex, "textures")
        assert vt.shape[0] == B and tex.shape[0] == B
        assert params.faces_textures.shape[-2] == nf
        assert params.faces_textures.ndim == 2 or params.faces_textures.shape[0] == B
        ft = _i32c(torch.as_tensor(params.faces_textures)).to(dev)
        nvt, H, W = vt.shape[1], tex.shape[2], tex.shape[3]
        _validate_indices(torch.as_tensor(params.faces_textures), nvt, "faces_textures")
        view_faces = view_faces or ft.ndim == 3
        if view_faces:
            ft = ft.expand(B, nf, 3).contiguous()
    if view_faces:
        # the kernels read row b of both index tensors for view b: the shared one is expanded (12 B nf bytes)
        faces_d = faces_d.expand(B, nf, 3).contiguous()
    cfg = _make_config(B, nv, nf, int(hyperparams.image_size),
                       _flags_of(hyperparams) | (_lib.NR_VIEW_FACES if view_faces else 0), hyperparams, nvt, H, W)
    light_pack = vn = None
    if hyperparams.draw_rgb and params.lights is not None:      # an empty list renders black, rasterize.py:252-283
        # shading: per-vertex normals by differentiable torch ops (O(nv + nf)), the per-pixel part in the kernels
        light_pack = light_lib.pack_lights(params.lights, B, dev)
        vn = light_lib.vertex_normals(vertices, faces_d, deterministic=bool(cfg.flags & _lib.NR_DETERMINISTIC))
    return cfg, faces_d, vt, ft, tex, vn, light_pack, bg


def rasterize_core(vertices, faces, params: RasterizeParam, hyperparams: RasterizeHyperparam):
    """``rasterize.py:194-329``. vertices [B,nv,3] screen space, faces [nf,3] or [B,nf,3] -> images [B,C,S,S]."""
    cfg, faces_d, vt, ft, tex, vn, light_pack, bg = _prepare(vertices, faces, params, hyperparams)
    light_types, light_data = light_pack if light_pack is not None else (None, None)
    return _Rasterize.apply(vertices, vt, tex, vn, bg, light_data, faces_d, ft, cfg, light_types)


def rasterize_maps(vertices, faces, params: RasterizeParam, hyperparams: RasterizeHyperparam):
    """Non-differentiable view of the internal maps the reference builds inside rasterize_core
    (``face_index_map`` :235, ``weight_map`` :236, depth :292) plus the images.  Test / debug aid."""
    cfg, faces_d, vt, ft, tex, vn, light_pack, bg = _prepare(vertices, faces, params, hyperparams)
    with torch.no_grad():
        images, internal, fim, wmap, dmap, _, _ = _forward_call(
            cfg, _f32c(vertices), faces_d, _f32c(vt) if vt is not None else None, ft,
            _f32c(tex) if tex is not None else None, True,
            (light_pack[0], _f32c(light_pack[1]), _f32c(vn)) if light_pack is not None else None,
            _f32c(bg) if bg is not None else None)
    return dict(images=images, internal_images=internal if internal is not None else images,
                face_index_map=fim, weight_map=wmap, depth_map=dmap)


def rasterize_silhouettes(vertices, faces, params: RasterizeParam, hyperparams: RasterizeHyperparam):
    hyperparams.draw_rgb = False
    hyperparams.draw_silhouettes = True
    hyperparams.draw_depth = False
    return rasterize_core(vertices, faces, params, hyperparams)[:, 0]


def rasterize_rgba(vertices, faces, params: RasterizeParam, hyperparams: RasterizeHyperparam):
    hyperparams.draw_rgb = True
    hyperparams.draw_silhouettes = True
    hyperparams.draw_depth = False
    return rasterize_core(vertices, faces, params, hyperparams)


def rasterize_rgb(vertices, faces, params: RasterizeParam, hyperparams: RasterizeHyperparam):
    hyperparams.draw_rgb = True
    hyperparams.draw_silhouettes = False
    hyperparams.draw_depth = False
    return rasterize_core(vertices, faces, params, hyperparams)


def rasterize_depth(vertices, faces, params: RasterizeParam, hyperparams: RasterizeHyperparam):
    hyperparams.draw_rgb = False
    hyperparams.draw_silhouettes = False
    hyperparams.draw_depth = True
    return rasterize_core(vertices, faces, params, hyperparams)[:, 0]


# ------------------------------------------------------------------------------------------------
# The two operators of the reference's pybind module, same names and argument order
# (cuda/rasterize_cuda.cpp:55-65, :81-90; called from rasterize.py:34-35 and :75).

def face_index_map_forward_safe(faces, face_index, num_faces, image_size, near, far, draw_backside,
                                eps, depth_min_delta):
    """faces [B,nf,3,3] CUDA f32 contiguous; face_index [B*S*S] CUDA i32, written in place and returned."""
    _require_cuda(faces, "faces")
    _require_cuda(face_index, "face_index")
    if not faces.is_contiguous():
        raise RuntimeError("faces must be contiguous")
    if not face_index.is_contiguous():
        raise RuntimeError("face_index must be contiguous")
    if faces.dtype != torch.float32 or face_index.dtype != torch.int32:
        raise RuntimeError("faces must be float32 and face_index int32")
    with torch.cuda.device(faces.device):
        stream = torch.cuda.current_stream(faces.device).cuda_stream
        rc = _lib.lib().nr_face_index_map_forward_safe(
            _ptr(faces), _ptr(face_index), faces.shape[0], int(num_faces), int(image_size), float(near),
            float(far), int(draw_backside), float(eps), float(depth_min_delta), ctypes.c_void_p(stream))
    _lib.check(rc, "face_index_map_forward_safe")
    return face_index


def compute_weight_map_c(faces, face_index_map, weight_map, num_faces, image_size):
    """faces [B,nf,3,3], face_index_map flat i32, weight_map [B*S*S,3] zeros written in place.
    Returns face_index_map like the reference (rasterize_cuda_kernel.cu:440)."""
    for t, n in ((faces, "faces"), (face_index_map, "face_index_map"), (weight_map, "weight_map")):
        _require_cuda(t, n)
        if not t.is_contiguous():
            raise RuntimeError("%s must be contiguous" % n)
    with torch.cuda.device(faces.device):
        stream = torch.cuda.current_stream(faces.device).cuda_stream
        rc = _lib.lib().nr_compute_weight_map(_ptr(faces), _ptr(face_index_map), _ptr(weight_map),
                                              faces.shape[0], int(num_faces), int(image_size),
                                              ctypes.c_void_p(stream))
    _lib.check(rc, "compute_weight_map_c")
    return face_index_map
