/*
 * nr_b200.h -- C ABI of the B200-native rasterize / sample / approximate-gradient path.
 *
 * This is the drop-in boundary.  The reference binds its native code through a pybind11
 * module (neural_renderer_torch/cuda/rasterize_cuda.cpp:93-99) whose live entry points are
 * face_index_map_forward_safe (:55-65) and compute_weight_map_c (:81-90); everything around
 * them is torch orchestration (neural_renderer_torch/rasterize.py:194-329) plus the
 * Differentiation autograd function (neural_renderer_torch/differentiation.py:6-40).
 * libnr_b200.so exports
 *   (1) the same two operators with the same argument meaning (nr_face_index_map_forward_safe,
 *       nr_compute_weight_map), and
 *   (2) the fused forward / backward of the whole path that rasterize_core drives
 *       (nr_rasterize_forward, nr_rasterize_backward, nr_rasterize_backward_lights,
 *       nr_differentiation_backward).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host; plain pointers and
 *     sizes only, no torch / ATen types;
 *   - the caller owns every buffer (as in the reference, rasterize.py:32-33,71); kernels
 *     write in place;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*) of the CURRENT device
 *     and the call returns without synchronising;
 *   - return value: NR_OK or an error code; nr_last_error() gives the message of the
 *     last failure on the calling thread.  CUDA launch errors are returned, not printf'd
 *     (the reference only prints them, rasterize_cuda_kernel.cu:386-388).
 *   - float tensors are float32, index tensors int32, layouts are C-contiguous.
 */
#ifndef NR_B200_H
#define NR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NR_ABI_VERSION 4

#if defined(__GNUC__)
#define NR_API __attribute__((visibility("default")))
#else
#define NR_API
#endif

enum {
    NR_OK = 0,
    NR_ERR_INVALID_ARGUMENT = 1,
    NR_ERR_CUDA = 2,
    NR_ERR_WORKSPACE_TOO_SMALL = 3
};

/* nrRasterConfig.flags */
#define NR_DRAW_RGB 1         /* rasterize.py:244-249  */
#define NR_DRAW_SILHOUETTES 2 /* rasterize.py:240-242  */
#define NR_DRAW_DEPTH 4       /* rasterize.py:290-292  */
#define NR_DRAW_BACKSIDE 8    /* rasterize_param.py:20 */
#define NR_ANTI_ALIASING 16   /* rasterize.py:227-228, 321-328 */
#define NR_DETERMINISTIC 32   /* backward: fixed-order reduction instead of float atomics */
#define NR_SPARSE_MAPS 128    /* forward: face_index_map / images_internal are only written where
                                 nr_rasterize_backward reads them (non-empty 16x16 tiles; for images_internal
                                 also the empty tiles next to one).  `images` is always complete.  Needs the forward's
                                 tile_list passed on to the backward. */
#define NR_FINE_TILES 256     /* forward: bin into 8x8 instead of 16x16 tiles (general binning path).  For dense
                                 meshes (nrBinStats.max_tile_faces in the hundreds): lists four times shorter.
                                 tile_list is then in 8x8 units, [8 + 16 * B * ceil(R/8)^2] ints, and must NOT
                                 be passed to nr_rasterize_backward (pass NULL); NR_SPARSE_MAPS is ignored. */
#define NR_GENERAL_BINNING 64 /* forward: never take the one-kernel small-mesh binning path (see nrBinStats) */
#define NR_DENSE_RASTER 512   /* forward: meshes of SMALL triangles (nrBinStats.total_pairs of an earlier call >= ~32 per
                                 tile on average, a few tiles per face): no tile lists at all, one thread per face
                                 merging (depth, face) into a 64-bit global z-buffer with atomicMin, exact replay of
                                 the reference's sequential scan for contested pixels (nr_raster_zbuf.cu).  Same
                                 results bit for bit.  nr_workspace_bytes depends on this flag; nrBinStats then
                                 reports total_pairs = contested pixels, max_tile_faces = faces whose pixel box is
                                 above 4096 pixels (more than a few per cent of the faces: drop the flag),
                                 overflow = 1 when the candidate pool (pair_capacity / 4 entries) was too small
                                 (still exact, slower). */
#define NR_VIEW_FACES 1024    /* forward and backward: one mesh topology per view.  `faces` is [B, nf, 3] and, with
                                 NR_DRAW_RGB, `faces_textures` is [B, nf, 3] as well; view b reads row b of both.
                                 Views with fewer faces pad their rows with a degenerate face (three equal indices,
                                 e.g. 0 0 0): it is never drawn and gets no gradient.  faces must not be NULL. */

/* Mirrors RasterizeHyperparam (rasterize_param.py:13-33) plus the tensor extents. */
typedef struct nrRasterConfig {
    int32_t batch;            /* B: views */
    int32_t num_vertices;     /* nv */
    int32_t num_faces;        /* nf */
    int32_t image_size;       /* S: OUTPUT size; internal R = 2S with NR_ANTI_ALIASING */
    int32_t flags;            /* NR_DRAW_* | NR_ANTI_ALIASING | ... */
    float near_plane;         /* default 0.1   */
    float far_plane;          /* default 100   */
    float eps;                /* default 1e-5 (texture clamp, rasterize.py:121) */
    float depth_min_delta;    /* 1e-4, the z-test hysteresis (rasterize.py:35) */
    int32_t num_tex_vertices; /* nvt (0 when no texture) */
    int32_t tex_height;       /* H */
    int32_t tex_width;        /* W */
} nrRasterConfig;

/*
 * Optional shading inputs; NULL = unlit, black background.
 * Lights (rasterize.py:252-283 with the smooth normal map of :162-190), num_lights = 0 for none.
 * Light l of view b is data[(l * B + b) * 8 ..]: colour rgb, direction xyz, alpha, unused.
 * types[l]: 0 ambient (lights.py:22-24), 1 directional (:10-19), 2 specular (:27-39); +4 = backside
 * (|intensity| instead of relu).  vertex_normals [B, nv, 3] are the normalised per-vertex normals
 * (sum of the normals of the faces touching the vertex); the backward accumulates into
 * grad_vertex_normals [B, nv, 3] (caller zero-fills), from where autograd reaches the vertices.
 */
typedef struct nrLights {
    int32_t num_lights;
    const int32_t *types;        /* [L], device */
    const float *data;           /* [L, B, 8] */
    const float *vertex_normals; /* [B, nv, 3] */
    float *grad_vertex_normals;  /* backward only, may be NULL */
    /* Backgrounds [B, 3, R, R] at INTERNAL resolution, in output orientation: behind every background
     * pixel the rgb channels show backgrounds[b, :, Y, X] (2x2-averaged under anti-aliasing).  This is
     * what rasterize.py:156-159 intends (it fails on torch tensors); semantics follow the Chainer
     * original, neural_renderer_chainer/rasterize.py:574-577.  NULL = black. */
    const float *backgrounds;
} nrLights;

/*
 * Optional buffers the forward zero-fills while it rasterizes: the gradient accumulators of the
 * coming nr_rasterize_backward (which ADDS into its outputs).  The raster kernel is instruction-issue
 * bound and leaves HBM idle, so the fill costs nothing there; as a separate fill in front of the
 * backward it is a serial 30 MB write at BASELINE config 2.  ptr[i] 16-byte aligned, bytes[i] a
 * multiple of 4.  NULL / count 0 = nothing to fill.
 */
typedef struct nrZeroFill {
    int32_t count;               /* 0..4 */
    void *ptr[4];
    size_t bytes[4];
} nrZeroFill;

/*
 * Written by the forward into the workspace header and, when `stats_host` is given,
 * copied asynchronously to that (pinned) host struct so the caller can look at it once
 * `stats_event` has completed.  overflow != 0 means the (tile, face) pair list did not fit
 * `pair_capacity`: the results of that call are STILL CORRECT (the raster kernel then scans
 * every face of the view per pixel block, like the reference does) but slow; size the next
 * call's workspace for at least `total_pairs`.  No host synchronisation is ever required.
 */
typedef struct nrBinStats {
    int32_t total_pairs;      /* sum over tiles of faces whose pixel bbox touches the tile */
    int32_t max_tile_faces;   /* longest per-tile list */
    int32_t overflow;         /* 1: pair list longer than pair_capacity; 2: a view has more pairs than the
                                 one-kernel small-mesh binning holds in shared memory -> pass
                                 NR_GENERAL_BINNING from now on.  Results are correct either way. */
    int32_t bad_index;        /* bit 0: a face referenced a vertex outside [0, nv) (face dropped);
                                 bit 1: a face referenced a texture vertex outside [0, nvt) (its pixels are black,
                                 no gradient).  Both are an IndexError in the reference (rasterize.py:232,246). */
} nrBinStats;

NR_API int nr_abi_version(void);
NR_API const char *nr_last_error(void);

/* Number of channels the configuration renders: 3*rgb + silhouettes + depth. */
NR_API int nr_num_channels(int32_t flags);

/* Thin wrappers so a host without a CUDA binding (ctypes, cgo ...) can wait for the statistics. */
NR_API int nr_event_create(void **event);
NR_API int nr_event_destroy(void *event);
NR_API int nr_event_synchronize(void *event);
NR_API int nr_event_query(void *event); /* 1 complete, 0 not yet, -1 error */

/*
 * Per-kernel timing hook for bench.py: while enabled, every kernel this library launches is
 * bracketed by CUDA events on its launch stream.  nr_profile_collect synchronises those events and
 * ADDS the elapsed milliseconds / launch counts per slot into ms[NR_PROF_SLOTS] / launches[...]
 * (slots: 0 memset, 1 setup_count, 2 scan_tiles, 3 scatter, 4 sort_long, 5 raster, 6 backward,
 * 7 differentiation_backward, 8 weight_map_compat, 9 zbuf_faces, 10 camera_forward, 11 camera_backward,
 * 12 zbuf_resolve, 13 zbuf_shade), then forgets them.
 */
#define NR_PROF_SLOTS 14
NR_API int nr_profile_enable(int on);
NR_API int nr_profile_collect(float *ms, int32_t *launches);

/* Bytes of zero-filled scratch the deterministic backward needs. */
NR_API size_t nr_deterministic_scratch_bytes(const nrRasterConfig *cfg);

/* Bytes of scratch the forward needs for `pair_capacity` (tile, face) pairs. */
NR_API size_t nr_workspace_bytes(const nrRasterConfig *cfg, int64_t pair_capacity);

/*
 * Fused forward of rasterize_core (rasterize.py:194-329); lights / backgrounds through nrLights:
 * face gather (:232), z-buffer (:235), weight map (:236), texture sampling (:249),
 * silhouettes (:242), depth (:292), channel merge (:295-310), permute + flip (:315-316),
 * 2x2 anti-aliasing mean (:321-328).
 *
 *   vertices            [B, nv, 3]   screen-space x, y in [-1, 1], z = depth
 *   faces               [nf, 3]      vertex ids; NULL means face f uses vertices 3f, 3f+1, 3f+2
 *                                    (i.e. `vertices` is the gathered [B, nf, 3, 3] tensor);
 *                                    [B, nf, 3] with NR_VIEW_FACES
 *   vertices_textures   [B, nvt, 2]  texel coordinates           (NR_DRAW_RGB only)
 *   faces_textures      [nf, 3]      ids into vertices_textures  (NR_DRAW_RGB only; [B, nf, 3] with NR_VIEW_FACES)
 *   textures            [B, 3, H, W]                             (NR_DRAW_RGB only)
 *   face_index_map      [B, R, R]    out, -1 on background (never NULL)
 *   weight_map          [B, R, R, 3] out, optional (NULL to skip)
 *   depth_map           [B, R, R]    out, optional (NULL to skip); 1/sum(w/z), 0 on background
 *   images              [B, C, S, S] out, channel order rgb, silhouette, depth
 *   images_internal     [B, C, R, R] out, required with NR_ANTI_ALIASING (the backward
 *                                    stencil runs at internal resolution), else may be NULL
 *                                    (then `images` itself is the internal image)
 *   aux_map             [B, R, R, 6] with NR_DRAW_RGB, else [B, R, R, 3]: out, optional (NULL to skip), 8-byte
 *                       aligned.  Forward -> backward state, written at FOREGROUND pixels only (not initialised
 *                       elsewhere): the normalised weights w0 w1 w2 and, with colour, the three quotients of the
 *                       perspective-correct texel coordinate (rasterize.py:113-119: depth, sum w u / z, sum w v / z).
 *                       Handed to nr_rasterize_backward it saves that kernel 9 scattered vertex loads and 12 IEEE
 *                       divisions per pixel (the forward has the values in registers anyway).
 *   tile_list           [8 + 16 * B * ceil(R/16)^2] i32 out, optional, 16-byte aligned: the non-empty
 *                       16x16 tiles in four length classes (longest face lists first); elements 0..3
 *                       = entries per class, then 4 ints per tile (view, tile_x | tile_y << 16, list
 *                       offset, list length), class k starting at entry k * B * tiles.  Pass it to
 *                       nr_rasterize_backward so the backward visits only those tiles.
 *   workspace           nr_workspace_bytes(cfg, pair_capacity) bytes, 256-byte aligned
 *   stats_host          optional pinned host nrBinStats
 *   stats_event         optional cudaEvent_t (as void*, e.g. from nr_event_create) recorded right
 *                       after the stats copy, which follows the raster kernel (bad_index bit 1 is set there)
 *   zero_fill           optional, see nrZeroFill
 *
 * Every element of face_index_map / images / images_internal is written (empty tiles and background
 * pixels by the raster kernel itself): the caller does not initialise them.  With NR_SPARSE_MAPS the two
 * maps that only the backward consumes are left untouched where it never looks.
 */
NR_API int nr_rasterize_forward(const nrRasterConfig *cfg, const float *vertices, const int32_t *faces,
                         const float *vertices_textures, const int32_t *faces_textures,
                         const float *textures, int32_t *face_index_map, float *weight_map,
                         float *depth_map, float *images, float *images_internal, float *aux_map,
                         int32_t *tile_list, void *workspace, size_t workspace_bytes, int64_t pair_capacity,
                         nrBinStats *stats_host, void *stats_event, const nrZeroFill *zero_fill,
                         const nrLights *lights, void *stream);

/*
 * Fused backward: AA / flip / permute backward, the Differentiation stencil
 * (differentiation.py:13-36 with utils.py:75-101), coordinate_map -> faces -> vertices
 * scatter (autograd of rasterize.py:91-97,232), sample_textures backward (:100-153) into
 * textures, face z and vertices_textures, and depth-map backward (:80-88).
 *
 *   face_index_map      [B, R, R]    from the forward
 *   images_internal     [B, C, R, R] from the forward (pass `images` when not anti-aliased)
 *   aux_map             from the forward, or NULL (weights and texel coordinates are then recomputed; always so
 *                       with NR_DETERMINISTIC)
 *   tile_list           from the forward, or NULL (then every tile is visited)
 *   grad_images         [B, C, S, S] upstream gradient
 *   grad_vertices       [B, nv, 3]   out, ACCUMULATED into (caller zero-fills)
 *   grad_textures       [B, 3, H, W] out, accumulated, optional
 *   grad_vertices_textures [B, nvt, 2] out, accumulated, optional
 *   deterministic_scratch  only with NR_DETERMINISTIC in cfg->flags: nr_deterministic_scratch_bytes(cfg)
 *                       zero-filled bytes.  Contributions are then rounded once to 64-bit fixed point
 *                       and summed with integer atomics, so the gradients are bit-identical from run to run
 *                       (float atomics depend on arrival order).  The unit is chosen per view on the device:
 *                       2^(E_b - 32), with m_b = max |grad_images| over view b's finite values in
 *                       [2^(E_b - 1), 2^E_b) (E_b = 0 for an all-zero view).  So the resolution is
 *                       <= 4.7e-10 m_b and the results are valid while every |sum| < 2^(31 + E_b) (>= 2.1e9 m_b);
 *                       scaling G by a power of two scales the gradients exactly, and a view's bits do not
 *                       depend on the other views of the call.  NaN and +-inf contributions are summed as floats
 *                       and come out as with float atomics.  Covers grad_vertex_normals and grad_light_data.
 */
NR_API int nr_rasterize_backward(const nrRasterConfig *cfg, const float *vertices, const int32_t *faces,
                          const float *vertices_textures, const int32_t *faces_textures,
                          const float *textures, const int32_t *face_index_map,
                          const float *images_internal, const float *aux_map, const int32_t *tile_list,
                          const float *grad_images, float *grad_vertices, float *grad_textures,
                          float *grad_vertices_textures, void *deterministic_scratch, const nrLights *lights,
                          void *stream);

/*
 * nr_rasterize_backward plus the gradient with respect to the light data (autograd of rasterize.py:256-283
 * with respect to each light's color, direction and alpha).  nr_rasterize_backward is this call with
 * grad_light_data = light_deterministic_scratch = NULL.
 *
 *   grad_light_data     [L, B, 8] out, ACCUMULATED into, in the layout of nrLights.data: colour 0..2,
 *                       direction 3..5 (directional lights only), alpha 6 (specular lights only); the other slots
 *                       are left as they are.  NULL = not wanted (no extra work).  Only lit colour calls
 *                       (NR_DRAW_RGB and lights->num_lights > 0) have a light gradient; otherwise it is left as is.
 *   light_deterministic_scratch  only with NR_DETERMINISTIC and a non-NULL grad_light_data: L * B * 8 zero-filled
 *                       int64 (8-byte aligned); the light gradient is then bit-identical from run to run too.
 * The per-pixel terms are summed per warp in registers (a fixed order), so each warp of a tile adds at most one
 * value per (light, parameter).
 */
NR_API int nr_rasterize_backward_lights(const nrRasterConfig *cfg, const float *vertices, const int32_t *faces,
                                 const float *vertices_textures, const int32_t *faces_textures,
                                 const float *textures, const int32_t *face_index_map,
                                 const float *images_internal, const float *aux_map, const int32_t *tile_list,
                                 const float *grad_images, float *grad_vertices, float *grad_textures,
                                 float *grad_vertices_textures, void *deterministic_scratch, const nrLights *lights,
                                 float *grad_light_data, void *light_deterministic_scratch, void *stream);

/*
 * Differentiation.backward (differentiation.py:13-36) on channels-last tensors, as the
 * public differentiation(images, coordinates) op sees them:
 *   images, grad_output [B, R, R, C] -> grad_coordinates [B, R, R, 2] (x, y), overwritten.
 */
NR_API int nr_differentiation_backward(const float *images, const float *grad_output,
                                float *grad_coordinates, int32_t batch, int32_t image_size,
                                int32_t channels, void *stream);

/*
 * Fused camera transform (look_at.py:28-42 + perspective.py:9-17): out = persp(R (v - eye)).
 *   vertices [B, nv, 3] world space, rotation [B, 3, 3] (rows = camera x, y, z axes), eye [B, 3]
 *   out [B, nv, 3] screen space; perspective != 0 divides x and y by z and by width = tan(angle).
 *   shared_mesh != 0: `vertices` is ONE mesh [1, nv, 3] seen by all B cameras (the reference gets the same by
 *   broadcasting, look_at.py:41; multi-view optimisation, examples_pytorch/example2.py).
 * Backward: grad_vertices [B, nv, 3] is written - with shared_mesh [1, nv, 3], the sum over the B views in
 * view order (deterministic; no [B, nv, 3] intermediate, no separate reduction); partial
 * [B, nr_camera_partial_blocks(nv), 12] receives per-block sums of d loss / d rotation (9, row-major) and
 * d loss / d eye (3) - sum them over dim 1 - or is NULL when the cameras need no gradient.
 */
NR_API int nr_camera_partial_blocks(int32_t num_vertices);
NR_API int nr_camera_forward(const float *vertices, const float *rotation, const float *eye, float *out,
                             int32_t batch, int32_t num_vertices, int32_t perspective, float width,
                             int32_t shared_mesh, void *stream);
NR_API int nr_camera_backward(const float *vertices, const float *rotation, const float *eye,
                              const float *grad_out, float *grad_vertices, float *partial, int32_t batch,
                              int32_t num_vertices, int32_t perspective, float width, int32_t shared_mesh,
                              void *stream);

/*
 * Shared mesh on several GPUs of one box (BASELINE config 3: multi-view optimisation, 8 views per GPU): the
 * shared-mesh camera backward FUSED with the all-reduce of its [1, nv, 3] result over NVLink peer memory - no
 * NCCL call, no second kernel.  Every rank passes the same `peer_buffers`: world pointers, entry r = rank r's
 * exchange buffer of nr_camera_exchange_bytes(nv, world) bytes as mapped into THIS process (symmetric memory /
 * CUDA IPC; zero-filled once before the first call, then owned by these calls), and its own `epoch` (four ints of
 * device memory, zero-filled once; epoch[2] becomes 1 if a peer failed to show up within a few seconds).  A thread
 * sums its vertex over the local views, pushes the three sums into its slots of every peer's buffer as 8-byte
 * (value, epoch) words - written atomically, so no flag and no fence is needed: NCCL's LL trade - polls its own
 * buffer for the words of every peer, adds them in rank order and writes grad_vertices: bit-identical on every
 * rank and from run to run.  All ranks
 * must call it the same number of times (it is a collective).  The grid must be resident as a whole
 * (nv <= 256 * SMs * resident CTAs per SM: otherwise NR_ERR_INVALID_ARGUMENT, use NCCL).
 */
NR_API int nr_camera_exchange_bytes(int32_t num_vertices, int32_t world);
NR_API int nr_camera_backward_shared_allreduce(const float *vertices, const float *rotation, const float *eye,
                                               const float *grad_out, float *grad_vertices, float *partial,
                                               int32_t batch, int32_t num_vertices, int32_t perspective, float width,
                                               int32_t rank, int32_t world, void *const *peer_buffers,
                                               int32_t *epoch, void *stream);

/*
 * Same operator as face_index_map_forward_safe (rasterize_cuda.cpp:55-65):
 *   faces [B, nf, 3, 3], face_index [B*S*S] written in place (pre-fill not required).
 * `eps` is accepted and unused, like in the reference kernel.  Like the reference operator the call is
 * ASYNCHRONOUS: it enqueues on `stream` and returns.  Scratch comes from a per (device, stream) cache owned by
 * the library, sized from the statistics of the previous calls on that stream (read when their event has
 * completed, never waited for); a call whose pair list outgrows the scratch is still exact (device-side
 * fallback, see nrBinStats) and the next one gets a larger scratch.  The only host synchronisation is a
 * cudaStreamSynchronize(stream) in front of a scratch REallocation (growth), i.e. in the first call(s) of a shape.
 */
NR_API int nr_face_index_map_forward_safe(const float *faces, int32_t *face_index, int32_t batch,
                                   int32_t num_faces, int32_t image_size, float near_plane,
                                   float far_plane, int32_t draw_backside, float eps,
                                   float depth_min_delta, void *stream);

/*
 * Same operator as compute_weight_map_c (rasterize_cuda.cpp:81-90):
 *   faces [B, nf, 3, 3], face_index_map [B*S*S], weight_map [B*S*S, 3]; only foreground
 *   pixels are written (the caller zero-fills, rasterize.py:71).
 */
NR_API int nr_compute_weight_map(const float *faces, const int32_t *face_index_map, float *weight_map,
                          int32_t batch, int32_t num_faces, int32_t image_size, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* NR_B200_H */
