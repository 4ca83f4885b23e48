// nr_abi.cu -- extern "C" entry points declared in include/nr_b200.h.
#include <cstdlib>
#include <stdio.h>
#include <string.h>

#include <mutex>

#include "../../include/nr_b200.h"
#include "nr_kernels.h"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, const char *detail = "") {
    snprintf(g_err, sizeof(g_err), fmt, detail);
    return code;
}
int fail_cuda(cudaError_t e, const char *where) {
    snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
    return NR_ERR_CUDA;
}

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct Carve {
    nr::BinHeader *hdr;
    int *tile_count, *tile_offset, *tile_cursor;
    nr::FaceRec *rec;
    int32_t *pairs;
    int32_t *tile_list;
    // z-buffer path (NR_DENSE_RASTER)
    unsigned *zb_bitmap, *zb_coarse;
    uint2 *zb_box;
    unsigned long long *zbuf;
    int *zb_head, *zb_pix_of;
    int4 *zb_nodes;
    int zb_wpr, zb_crows, zb_slot_cap, zb_node_cap;
    size_t bytes;
};

// NR_DENSE_RASTER: header | contested-pixel bitmap (adjacent: one memset clears both) | z-buffer | list heads |
// pixel of every slot | candidate nodes | tile list.  pair_capacity counts 4-byte units as in the tile pipeline:
// a quarter of it is the number of 16-byte candidate nodes (and of contested pixels) the call can hold.
Carve carve_dense(void *base, int B, int nf, int R, long long pair_capacity) {
    const int ntx = (R + nr::TILE - 1) / nr::TILE;
    const size_t nt = (size_t)B * ntx * ntx;
    char *p = (char *)base;
    size_t off = 0;
    Carve c;
    memset(&c, 0, sizeof(c));
    c.hdr = (nr::BinHeader *)(p + off);
    off += sizeof(nr::BinHeader);
    c.zb_wpr = (R + 31) / 32;
    c.zb_crows = (R + 7) / 8;
    c.zb_bitmap = (unsigned *)(p + off);
    off += (size_t)B * R * c.zb_wpr * sizeof(unsigned);
    c.zb_coarse = (unsigned *)(p + off);
    off = align256(off + (size_t)B * c.zb_crows * c.zb_wpr * sizeof(unsigned));
    c.zb_box = (uint2 *)(p + off);
    off = align256(off + (size_t)B * nf * sizeof(uint2));
    c.zbuf = (unsigned long long *)(p + off);
    off = align256(off + (size_t)B * R * R * sizeof(unsigned long long));
    long long cap = pair_capacity / 4;
    if (cap < 1024) cap = 1024;
    if (cap > 0x3fffffffLL) cap = 0x3fffffffLL;
    c.zb_slot_cap = c.zb_node_cap = (int)cap;
    c.zb_head = (int *)(p + off);
    off = align256(off + (size_t)cap * sizeof(int));
    c.zb_pix_of = (int *)(p + off);
    off = align256(off + (size_t)cap * sizeof(int));
    c.zb_nodes = (int4 *)(p + off);
    off = align256(off + (size_t)cap * sizeof(int4));
    c.tile_list = (int32_t *)(p + off);
    off = align256(off + (nr::TILE_LIST_HDR + nr::TILE_ENTRY_INTS * nr::TILE_CLASSES * nt) * sizeof(int32_t));
    c.bytes = off;
    return c;
}

// header and tile_count must be adjacent (one memset clears both)
Carve carve(void *base, int B, int nf, int R, long long pair_capacity, int tile) {
    const int ntx = (R + tile - 1) / tile;
    const size_t nt = (size_t)B * ntx * ntx;
    char *p = (char *)base;
    size_t off = 0;
    Carve c;
    memset(&c, 0, sizeof(c));
    c.hdr = (nr::BinHeader *)(p + off);
    off += sizeof(nr::BinHeader);
    c.tile_count = (int *)(p + off);
    off = align256(off + nt * sizeof(int));
    c.tile_offset = (int *)(p + off);
    off = align256(off + nt * sizeof(int));
    c.tile_cursor = (int *)(p + off);
    off = align256(off + nt * sizeof(int));
    c.rec = (nr::FaceRec *)(p + off);
    off = align256(off + (size_t)B * nf * sizeof(nr::FaceRec));
    c.pairs = (int32_t *)(p + off);
    off = align256(off + (size_t)(pair_capacity > 0 ? pair_capacity : 1) * sizeof(int32_t));
    c.tile_list = (int32_t *)(p + off);
    off = align256(off + (nr::TILE_LIST_HDR + nr::TILE_ENTRY_INTS * nr::TILE_CLASSES * nt) * sizeof(int32_t));
    c.bytes = off;
    return c;
}

int sm_count_cached() {
    static int cached[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (!cached[dev]) {
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        cached[dev] = n > 0 ? n : 148;
    }
    return cached[dev];
}

// tile edge of the binning: 16, or 8 with NR_FINE_TILES (which implies the general binning path)
int tile_edge(const nrRasterConfig *cfg) {
    return ((cfg->flags & NR_FINE_TILES) && !(cfg->flags & NR_DENSE_RASTER)) ? nr::FINE_TILE : nr::TILE;
}

// ints from one view's face rows to the next: every view reads the same [nf, 3] rows, or its own of [B, nf, 3]
int view_face_stride(const nrRasterConfig *cfg) {
    return (cfg->flags & NR_VIEW_FACES) ? 3 * cfg->num_faces : 0;
}

// texture elements of one view: [3, H, W], or with NR_FACE_TEXTURES the per-face cubes [nf, ts, ts, ts, 3] (H = W = ts)
size_t tex_elems_per_view(const nrRasterConfig *cfg) {
    if (cfg->flags & NR_FACE_TEXTURES) {
        const size_t ts = cfg->tex_height > 0 ? (size_t)cfg->tex_height : 0;
        return (size_t)(cfg->num_faces > 0 ? cfg->num_faces : 0) * ts * ts * ts * 3;
    }
    return (size_t)3 * cfg->tex_height * cfg->tex_width;
}

int check_config(const nrRasterConfig *cfg) {
    if (!cfg) return fail(NR_ERR_INVALID_ARGUMENT, "config is NULL");
    if (cfg->batch < 0 || cfg->num_vertices < 0 || cfg->num_faces < 0 || cfg->image_size <= 0)
        return fail(NR_ERR_INVALID_ARGUMENT, "negative extent or image_size <= 0");
    if (cfg->batch > 65535) return fail(NR_ERR_INVALID_ARGUMENT, "batch > 65535");
    if ((cfg->flags & NR_VIEW_FACES) && cfg->num_faces > 0x7fffffff / 3)
        return fail(NR_ERR_INVALID_ARGUMENT, "NR_VIEW_FACES: a view's face rows exceed 2^31 ints");
    const long long R = (long long)cfg->image_size * ((cfg->flags & NR_ANTI_ALIASING) ? 2 : 1);
    if (R > 32768) return fail(NR_ERR_INVALID_ARGUMENT, "internal resolution > 32768");
    if (!(cfg->flags & (NR_DRAW_RGB | NR_DRAW_SILHOUETTES | NR_DRAW_DEPTH)))
        return fail(NR_ERR_INVALID_ARGUMENT, "nothing to draw: no NR_DRAW_* flag");
    if (cfg->flags & NR_FACE_TEXTURES) {
        if (!(cfg->flags & NR_DRAW_RGB)) return fail(NR_ERR_INVALID_ARGUMENT, "NR_FACE_TEXTURES needs NR_DRAW_RGB");
        if (cfg->tex_height < 1 || cfg->tex_width != cfg->tex_height || cfg->num_tex_vertices != 0)
            return fail(NR_ERR_INVALID_ARGUMENT, "NR_FACE_TEXTURES needs tex_height = tex_width = ts >= 1 and num_tex_vertices = 0");
        // the kernels address a view's cubes with 32-bit offsets
        const long long ts = cfg->tex_height;
        if (ts > 1290 || (long long)cfg->num_faces * ts * ts * ts * 3 >= (1ll << 31))
            return fail(NR_ERR_INVALID_ARGUMENT, "NR_FACE_TEXTURES: nf * ts^3 * 3 of one view must be below 2^31");
    }
    return NR_OK;
}

// scratch of the reference-signature operator, one per (device, stream): the operator is asynchronous, so two
// streams must not share a workspace
struct CompatScratch {
    int device = -1;
    cudaStream_t stream = nullptr;
    void *ptr = nullptr;
    size_t bytes = 0;
    long long pair_capacity = 0;
    nrBinStats *stats_host = nullptr;    // pinned; written by the copy that follows the raster kernel
    cudaEvent_t stats_event = nullptr;
    bool pending = false;                // a call whose statistics have not been read yet
    int pend_faces = 0, pend_size = 0;   // its shape
    int general_faces = -1, general_size = -1;   // this shape outgrew the one-kernel binning (nrBinStats.overflow == 2)
    unsigned long long last_use = 0;
};
std::mutex g_compat_mu;
constexpr int COMPAT_SLOTS = 32;
CompatScratch g_compat[COMPAT_SLOTS];
unsigned long long g_compat_clock = 0;

}  // namespace

extern "C" {

int nr_abi_version(void) { return NR_ABI_VERSION; }
const char *nr_last_error(void) { return g_err; }

int nr_num_channels(int32_t flags) {
    return ((flags & NR_DRAW_RGB) ? 3 : 0) + ((flags & NR_DRAW_SILHOUETTES) ? 1 : 0) +
           ((flags & NR_DRAW_DEPTH) ? 1 : 0);
}

int nr_event_create(void **event) {
    if (!event) return fail(NR_ERR_INVALID_ARGUMENT, "event is NULL");
    cudaEvent_t ev;
    cudaError_t e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e != cudaSuccess) return fail_cuda(e, "cudaEventCreate");
    *event = (void *)ev;
    return NR_OK;
}
int nr_event_destroy(void *event) {
    if (!event) return NR_OK;
    cudaError_t e = cudaEventDestroy((cudaEvent_t)event);
    return e == cudaSuccess ? NR_OK : fail_cuda(e, "cudaEventDestroy");
}
int nr_event_query(void *event) {
    if (!event) return -1;
    cudaError_t e = cudaEventQuery((cudaEvent_t)event);
    if (e == cudaSuccess) return 1;
    if (e == cudaErrorNotReady) return 0;
    fail_cuda(e, "cudaEventQuery");
    return -1;
}
int nr_event_synchronize(void *event) {
    if (!event) return fail(NR_ERR_INVALID_ARGUMENT, "event is NULL");
    cudaError_t e = cudaEventSynchronize((cudaEvent_t)event);
    return e == cudaSuccess ? NR_OK : fail_cuda(e, "cudaEventSynchronize");
}

// 64-bit accumulators of the deterministic scratch: vertices, textures, vertices_textures, vertex normals (lights),
// back to back.  The B per-view maxima of |grad_images| (BackwardArgs::det_gmax) follow them.
static size_t det_fixed_elems(const nrRasterConfig *cfg) {
    return (size_t)cfg->batch * cfg->num_vertices * 3 +
           (size_t)cfg->batch * tex_elems_per_view(cfg) +
           (size_t)cfg->batch * cfg->num_tex_vertices * 2 +
           (size_t)cfg->batch * cfg->num_vertices * 3;
}

size_t nr_deterministic_scratch_bytes(const nrRasterConfig *cfg) {
    if (!cfg) return 0;
    return det_fixed_elems(cfg) * sizeof(long long) + (((size_t)cfg->batch * sizeof(unsigned) + 7) & ~(size_t)7);
}

size_t nr_workspace_bytes(const nrRasterConfig *cfg, int64_t pair_capacity) {
    if (!cfg) return 0;
    const int R = cfg->image_size * ((cfg->flags & NR_ANTI_ALIASING) ? 2 : 1);
    if (cfg->flags & NR_DENSE_RASTER) return carve_dense(nullptr, cfg->batch, cfg->num_faces, R, pair_capacity).bytes;
    return carve(nullptr, cfg->batch, cfg->num_faces, R, pair_capacity, tile_edge(cfg)).bytes;
}

int nr_rasterize_forward(const nrRasterConfig *cfg, const float *vertices, const int32_t *faces,
                         const float *vertices_textures, const int32_t *faces_textures,
                         const float *textures, int32_t *face_index_map, float *weight_map,
                         float *depth_map, float *images, float *images_internal, float *aux_map,
                         int32_t *tile_list, void *workspace, size_t workspace_bytes, int64_t pair_capacity,
                         nrBinStats *stats_host, void *stats_event, const nrZeroFill *zero_fill,
                         const nrLights *lights, void *stream_) {
    if (int rc = check_config(cfg)) return rc;
    cudaStream_t stream = (cudaStream_t)stream_;
    const bool aa = cfg->flags & NR_ANTI_ALIASING, rgb = cfg->flags & NR_DRAW_RGB;
    const int R = cfg->image_size * (aa ? 2 : 1);
    if (!vertices && cfg->batch * cfg->num_faces > 0) return fail(NR_ERR_INVALID_ARGUMENT, "vertices is NULL");
    if (!face_index_map) return fail(NR_ERR_INVALID_ARGUMENT, "face_index_map is NULL");
    if ((cfg->flags & NR_VIEW_FACES) && !faces) return fail(NR_ERR_INVALID_ARGUMENT, "NR_VIEW_FACES needs faces [B, nf, 3]");
    const bool cube = (cfg->flags & NR_FACE_TEXTURES) != 0;
    if (cube && (vertices_textures || faces_textures || !textures))
        return fail(NR_ERR_INVALID_ARGUMENT, "NR_FACE_TEXTURES needs textures [B, nf, ts, ts, ts, 3] and NULL vertices_textures / faces_textures");
    if (cube && aux_map) return fail(NR_ERR_INVALID_ARGUMENT, "NR_FACE_TEXTURES: no aux_map in this mode");
    if (rgb && !cube && (!vertices_textures || !faces_textures || !textures))
        return fail(NR_ERR_INVALID_ARGUMENT, "NR_DRAW_RGB needs vertices_textures, faces_textures and textures");
    if (rgb && !cube && (cfg->tex_height <= 0 || cfg->tex_width <= 0 || cfg->num_tex_vertices <= 0))
        return fail(NR_ERR_INVALID_ARGUMENT, "NR_DRAW_RGB needs positive texture extents");
    if (images && aa && !images_internal)
        return fail(NR_ERR_INVALID_ARGUMENT, "anti-aliasing needs images_internal");
    if (!workspace || ((uintptr_t)workspace & 255)) return fail(NR_ERR_INVALID_ARGUMENT, "workspace NULL or not 256-byte aligned");
    if (pair_capacity < 0 || pair_capacity > 0x7fffffffLL) return fail(NR_ERR_INVALID_ARGUMENT, "pair_capacity out of range");
    const int tile = tile_edge(cfg);
    {
        // work items (warp blocks of all tiles, fill chunks) are counted in 32-bit integers
        const long long ntx_ = (R + tile - 1) / tile;
        if ((long long)cfg->batch * ntx_ * ntx_ * 8 > 0x3fffffffLL || (long long)cfg->batch * cfg->num_faces > 0x7fffffffLL)
            return fail(NR_ERR_INVALID_ARGUMENT, "batch x tiles (or batch x faces) too large for one call: split the batch");
    }
    const bool dense = (cfg->flags & NR_DENSE_RASTER) != 0;
    if (dense && (long long)cfg->batch * R * R > 0x7fffffffLL)
        return fail(NR_ERR_INVALID_ARGUMENT, "NR_DENSE_RASTER: batch x pixels too large for one call: split the batch");
    // (k_zb_faces keeps two flag bits above a face index)
    if (dense && cfg->num_faces >= (1 << 29))
        return fail(NR_ERR_INVALID_ARGUMENT, "NR_DENSE_RASTER: more than 2^29 faces per view");
    const Carve c = dense ? carve_dense(workspace, cfg->batch, cfg->num_faces, R, pair_capacity)
                          : carve(workspace, cfg->batch, cfg->num_faces, R, pair_capacity, tile);
    if (c.bytes > workspace_bytes) return fail(NR_ERR_WORKSPACE_TOO_SMALL, "workspace smaller than nr_workspace_bytes()");
    if (cfg->batch == 0) return NR_OK;

    nr::BinningArgs ba;
    ba.verts = vertices;
    ba.faces = faces;
    ba.face_stride = view_face_stride(cfg);
    ba.B = cfg->batch;
    ba.nv = cfg->num_vertices;
    ba.nf = cfg->num_faces;
    ba.R = R;
    ba.draw_backside = (cfg->flags & NR_DRAW_BACKSIDE) ? 1 : 0;
    ba.ntx = (R + tile - 1) / tile;
    ba.tile_shift = tile == nr::TILE ? 4 : 3;
    ba.rec = c.rec;
    ba.tile_count = c.tile_count;
    ba.tile_offset = c.tile_offset;
    ba.tile_cursor = c.tile_cursor;
    ba.pairs = c.pairs;
    ba.pair_capacity = pair_capacity;
    ba.hdr = c.hdr;
    ba.tile_list = tile_list ? tile_list : c.tile_list;
    ba.sm_count = sm_count_cached();
    ba.one_cta_per_view = (cfg->flags & (NR_GENERAL_BINNING | NR_FINE_TILES | NR_DENSE_RASTER)) ? 0 : 1;

    nr::RasterArgs ra;
    ra.rec = c.rec;
    ra.tile_count = c.tile_count;
    ra.tile_offset = c.tile_offset;
    ra.pairs = c.pairs;
    ra.hdr = c.hdr;
    ra.tile_list = ba.tile_list;
    ra.sm_count = ba.sm_count;
    ra.B = cfg->batch;
    ra.nf = cfg->num_faces;
    ra.R = R;
    ra.S = cfg->image_size;
    ra.ntx = ba.ntx;
    ra.C = nr_num_channels(cfg->flags);
    ra.flags = cfg->flags;
    ra.near_plane = cfg->near_plane;
    ra.far_plane = cfg->far_plane;
    ra.eps = cfg->eps;
    ra.delta = cfg->depth_min_delta;
    ra.vt = vertices_textures;
    ra.ft = faces_textures;
    ra.tex = textures;
    ra.nvt = cfg->num_tex_vertices;
    ra.H = cfg->tex_height;
    ra.W = cfg->tex_width;
    ra.fim = face_index_map;
    ra.wmap = weight_map;
    ra.dmap = depth_map;
    ra.images = images;
    ra.internal = images_internal;
    if ((uintptr_t)aux_map & 7) return fail(NR_ERR_INVALID_ARGUMENT, "aux_map not 8-byte aligned");
    ra.aux = aux_map;
    ra.faces = faces;
    ra.face_stride = ba.face_stride;
    ra.nv = cfg->num_vertices;
    ra.verts = vertices;
    ra.zbuf = c.zbuf;
    ra.zb_bitmap = c.zb_bitmap;
    ra.zb_coarse = c.zb_coarse;
    ra.zb_box = c.zb_box;
    ra.zb_wpr = c.zb_wpr;
    ra.zb_crows = c.zb_crows;
    ra.zb_head = c.zb_head;
    ra.zb_pix_of = c.zb_pix_of;
    ra.zb_nodes = c.zb_nodes;
    ra.zb_slot_cap = c.zb_slot_cap;
    ra.zb_node_cap = c.zb_node_cap;
    ra.lights = nr::LightArgs{0, nullptr, nullptr, nullptr, nullptr, nullptr};
    if (lights && lights->num_lights > 0 && rgb) {
        if (!lights->types || !lights->data || !lights->vertex_normals)
            return fail(NR_ERR_INVALID_ARGUMENT, "lights: types, data and vertex_normals are required");
        ra.lights = nr::LightArgs{lights->num_lights, lights->types, lights->data, lights->vertex_normals, nullptr, nullptr};
    }
    if (lights && rgb) ra.lights.backgrounds = lights->backgrounds;

    ra.fine = tile != nr::TILE;
    // with 8x8 tiles the backward walks every 16x16 tile itself, so the maps must be complete
    ra.sparse_maps = ((cfg->flags & NR_SPARSE_MAPS) && !ra.fine) ? 1 : 0;
    ra.num_zero = 0;
    if (zero_fill) {
        if (zero_fill->count < 0 || zero_fill->count > 4) return fail(NR_ERR_INVALID_ARGUMENT, "zero_fill: count outside 0..4");
        for (int i = 0; i < zero_fill->count; ++i) {
            if (!zero_fill->ptr[i] || !zero_fill->bytes[i]) continue;
            if (((uintptr_t)zero_fill->ptr[i] & 15) || (zero_fill->bytes[i] & 3))
                return fail(NR_ERR_INVALID_ARGUMENT, "zero_fill: pointer not 16-byte aligned or size not a multiple of 4");
            ra.zero_ptr[ra.num_zero] = zero_fill->ptr[i];
            ra.zero_bytes[ra.num_zero++] = zero_fill->bytes[i];
        }
    }

    cudaError_t e;
    if ((e = nr::launch_background_fill(ra, stream)) != cudaSuccess) return fail_cuda(e, "map fill");
    if (dense) {
        e = nr::launch_raster_zbuf(ra, stream);
    } else {
        e = nr::launch_binning(ba, stream);
        if (e != cudaSuccess) return fail_cuda(e, "binning");
        e = nr::launch_raster(ra, stream);
    }
    if (e != cudaSuccess) return fail_cuda(e, "raster");
    if (stats_host) {
        e = cudaMemcpyAsync(stats_host, c.hdr, sizeof(nrBinStats), cudaMemcpyDeviceToHost, stream);
        if (e != cudaSuccess) return fail_cuda(e, "stats copy");
    }
    if (stats_event) {
        e = cudaEventRecord((cudaEvent_t)stats_event, stream);
        if (e != cudaSuccess) return fail_cuda(e, "stats event");
    }
    return NR_OK;
}

int nr_rasterize_backward(const nrRasterConfig *cfg, const float *vertices, const int32_t *faces,
                          const float *vertices_textures, const int32_t *faces_textures,
                          const float *textures, const int32_t *face_index_map,
                          const float *images_internal, const float *aux_map, const int32_t *tile_list,
                          const float *grad_images, float *grad_vertices, float *grad_textures,
                          float *grad_vertices_textures, void *deterministic_scratch, const nrLights *lights,
                          void *stream_) {
    return nr_rasterize_backward_lights(cfg, vertices, faces, vertices_textures, faces_textures, textures,
                                        face_index_map, images_internal, aux_map, tile_list, grad_images,
                                        grad_vertices, grad_textures, grad_vertices_textures, deterministic_scratch,
                                        lights, nullptr, nullptr, stream_);
}

int nr_rasterize_backward_lights(const nrRasterConfig *cfg, const float *vertices, const int32_t *faces,
                                 const float *vertices_textures, const int32_t *faces_textures,
                                 const float *textures, const int32_t *face_index_map,
                                 const float *images_internal, const float *aux_map, const int32_t *tile_list,
                                 const float *grad_images, float *grad_vertices, float *grad_textures,
                                 float *grad_vertices_textures, void *deterministic_scratch, const nrLights *lights,
                                 float *grad_light_data, void *light_deterministic_scratch, void *stream_) {
    if (int rc = check_config(cfg)) return rc;
    const bool aa = cfg->flags & NR_ANTI_ALIASING, rgb = cfg->flags & NR_DRAW_RGB;
    if (!vertices || !face_index_map || !images_internal || !grad_images || !grad_vertices)
        return fail(NR_ERR_INVALID_ARGUMENT, "backward: a required pointer is NULL");
    if ((cfg->flags & NR_VIEW_FACES) && !faces) return fail(NR_ERR_INVALID_ARGUMENT, "NR_VIEW_FACES needs faces [B, nf, 3]");
    const bool cube = (cfg->flags & NR_FACE_TEXTURES) != 0;
    if (cube && (vertices_textures || faces_textures || grad_vertices_textures || !textures))
        return fail(NR_ERR_INVALID_ARGUMENT, "NR_FACE_TEXTURES needs textures [B, nf, ts, ts, ts, 3] and NULL vertices_textures / faces_textures");
    if (cube && aux_map) return fail(NR_ERR_INVALID_ARGUMENT, "NR_FACE_TEXTURES: no aux_map in this mode");
    if (rgb && !cube && (!vertices_textures || !faces_textures || !textures))
        return fail(NR_ERR_INVALID_ARGUMENT, "NR_DRAW_RGB needs vertices_textures, faces_textures and textures");
    if (cfg->batch == 0) return NR_OK;
    nr::BackwardArgs a;
    a.verts = vertices;
    a.faces = faces;
    a.face_stride = view_face_stride(cfg);
    a.vt = vertices_textures;
    a.ft = faces_textures;
    a.tex = textures;
    a.fim = face_index_map;
    a.internal = images_internal;
    a.aux = (cfg->flags & NR_DETERMINISTIC) ? nullptr : aux_map;
    a.grad_images = grad_images;
    a.tile_list = tile_list;
    a.sm_count = sm_count_cached();
    a.grad_verts = grad_vertices;
    a.grad_tex = grad_textures;
    a.grad_vt = grad_vertices_textures;
    a.lights = nr::LightArgs{0, nullptr, nullptr, nullptr, nullptr, nullptr};
    if (lights && lights->num_lights > 0 && rgb) {
        if (!lights->types || !lights->data || !lights->vertex_normals)
            return fail(NR_ERR_INVALID_ARGUMENT, "lights: types, data and vertex_normals are required");
        a.lights = nr::LightArgs{lights->num_lights, lights->types, lights->data, lights->vertex_normals,
                                 lights->grad_vertex_normals, nullptr};
    }
    // without lights (or without colour) the light gradient is zero: nothing to add
    a.grad_light = a.lights.num > 0 ? grad_light_data : nullptr;
    a.det_light = nullptr;
    a.det_verts = a.det_tex = a.det_vt = a.det_vn = nullptr;
    a.det_gmax = nullptr;
    if (cfg->flags & NR_DETERMINISTIC) {
        if (!deterministic_scratch || ((uintptr_t)deterministic_scratch & 7))
            return fail(NR_ERR_INVALID_ARGUMENT, "NR_DETERMINISTIC needs deterministic_scratch (8-byte aligned, zero-filled)");
        long long *p = (long long *)deterministic_scratch;
        a.det_gmax = (unsigned *)(p + det_fixed_elems(cfg));
        a.det_verts = p;
        p += (size_t)cfg->batch * cfg->num_vertices * 3;
        if (grad_textures) {
            a.det_tex = p;
            p += (size_t)cfg->batch * tex_elems_per_view(cfg);
        }
        if (grad_vertices_textures) {
            a.det_vt = p;
            p += (size_t)cfg->batch * cfg->num_tex_vertices * 2;
        }
        if (a.lights.grad_vnormals) a.det_vn = p;
        if (a.grad_light) {
            if (!light_deterministic_scratch || ((uintptr_t)light_deterministic_scratch & 7))
                return fail(NR_ERR_INVALID_ARGUMENT,
                            "NR_DETERMINISTIC with grad_light_data needs light_deterministic_scratch (8-byte aligned, zero-filled)");
            a.det_light = (long long *)light_deterministic_scratch;
        }
    }
    a.B = cfg->batch;
    a.nv = cfg->num_vertices;
    a.nf = cfg->num_faces;
    a.S = cfg->image_size;
    a.R = cfg->image_size * (aa ? 2 : 1);
    a.ntx = (a.R + nr::TILE - 1) / nr::TILE;
    a.C = nr_num_channels(cfg->flags);
    a.flags = cfg->flags;
    a.nvt = cfg->num_tex_vertices;
    a.H = cfg->tex_height;
    a.W = cfg->tex_width;
    a.eps = cfg->eps;
    cudaError_t e = nr::launch_backward(a, (cudaStream_t)stream_);
    if (e != cudaSuccess) return fail_cuda(e, "backward");
    return NR_OK;
}

int nr_differentiation_backward(const float *images, const float *grad_output,
                                float *grad_coordinates, int32_t batch, int32_t image_size,
                                int32_t channels, void *stream_) {
    if (!images || !grad_output || !grad_coordinates)
        return fail(NR_ERR_INVALID_ARGUMENT, "differentiation: NULL pointer");
    if (batch < 0 || image_size <= 0 || channels <= 0)
        return fail(NR_ERR_INVALID_ARGUMENT, "differentiation: bad extents");
    cudaError_t e = nr::launch_differentiation_backward(images, grad_output, grad_coordinates, batch,
                                                        image_size, channels, (cudaStream_t)stream_);
    if (e != cudaSuccess) return fail_cuda(e, "differentiation backward");
    return NR_OK;
}

int nr_face_index_map_forward_safe(const float *faces, int32_t *face_index, int32_t batch,
                                   int32_t num_faces, int32_t image_size, float near_plane,
                                   float far_plane, int32_t draw_backside, float eps,
                                   float depth_min_delta, void *stream_) {
    (void)eps;   // unused by the reference kernel as well (rasterize_cuda_kernel.cu:61)
    if (!faces || !face_index) return fail(NR_ERR_INVALID_ARGUMENT, "faces / face_index is NULL");
    nrRasterConfig cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.batch = batch;
    cfg.num_vertices = num_faces * 3;
    cfg.num_faces = num_faces;
    cfg.image_size = image_size;
    cfg.flags = NR_DRAW_SILHOUETTES | (draw_backside ? NR_DRAW_BACKSIDE : 0);
    cfg.near_plane = near_plane;
    cfg.far_plane = far_plane;
    cfg.eps = 1e-5f;
    cfg.depth_min_delta = depth_min_delta;
    if (int rc = check_config(&cfg)) return rc;
    cudaStream_t stream = (cudaStream_t)stream_;

    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(g_compat_mu);
    // the scratch of this (device, stream); the least recently used slot is recycled when all are taken
    CompatScratch *sp = nullptr, *lru = &g_compat[0];
    for (CompatScratch &c : g_compat) {
        if (c.device == dev && c.stream == stream) { sp = &c; break; }
        if (c.last_use < lru->last_use) lru = &c;
    }
    if (!sp) {
        sp = lru;
        if (sp->device >= 0) {               // recycle: its work must have left the GPU before the memory goes
            int cur = dev;
            cudaSetDevice(sp->device);
            cudaStreamSynchronize(sp->stream);
            if (sp->ptr) cudaFree(sp->ptr);
            if (sp->stats_host) cudaFreeHost(sp->stats_host);
            if (sp->stats_event) cudaEventDestroy(sp->stats_event);
            cudaSetDevice(cur);
            (void)cudaGetLastError();
        }
        *sp = CompatScratch();
        sp->device = dev;
        sp->stream = stream;
    }
    CompatScratch &s = *sp;
    s.last_use = ++g_compat_clock;
    if (!s.stats_host) {
        cudaError_t e = cudaMallocHost((void **)&s.stats_host, sizeof(nrBinStats));
        if (e != cudaSuccess) return fail_cuda(e, "cudaMallocHost");
        memset(s.stats_host, 0, sizeof(nrBinStats));
        e = cudaEventCreateWithFlags(&s.stats_event, cudaEventDisableTiming);
        if (e != cudaSuccess) return fail_cuda(e, "cudaEventCreate");
    }
    // statistics of the previous call on this stream, if they have arrived (never waited for)
    if (s.pending && cudaEventQuery(s.stats_event) == cudaSuccess) {
        s.pending = false;
        if (s.stats_host->overflow) {
            const long long want = (long long)s.stats_host->total_pairs + (s.stats_host->total_pairs >> 2) + 1024;
            if (want > s.pair_capacity) s.pair_capacity = want;
            if (s.stats_host->overflow == 2) {
                s.general_faces = s.pend_faces;
                s.general_size = s.pend_size;
            }
        }
    }
    (void)cudaGetLastError();        // cudaErrorNotReady of the query is not an error
    long long cap = (long long)batch * num_faces * 4 + 1024;
    if (s.pair_capacity > cap) cap = s.pair_capacity;
    if (cap > 0x7fffffffLL) cap = 0x7fffffffLL;
    const size_t need = nr_workspace_bytes(&cfg, cap);
    if (need > s.bytes) {
        // growth: earlier calls on this stream may still use the old block
        cudaError_t e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) return fail_cuda(e, "face_index_map_forward_safe");
        if (s.ptr) cudaFree(s.ptr);
        s.ptr = nullptr;
        s.bytes = 0;
        s.pending = false;
        e = cudaMalloc(&s.ptr, need + need / 4);
        if (e != cudaSuccess) return fail_cuda(e, "cudaMalloc(scratch)");
        s.bytes = need + need / 4;
    }
    s.pair_capacity = cap;
    if (s.general_faces == num_faces && s.general_size == image_size) cfg.flags |= NR_GENERAL_BINNING;
    // the pinned statistics are owned by the call in flight until its event completes
    const bool track = !s.pending;
    int rc = nr_rasterize_forward(&cfg, faces, nullptr, nullptr, nullptr, nullptr, face_index, nullptr, nullptr, nullptr,
                                  nullptr, nullptr, nullptr, s.ptr, s.bytes, cap, track ? s.stats_host : nullptr,
                                  track ? (void *)s.stats_event : nullptr, nullptr, nullptr, stream);
    if (rc != NR_OK) return rc;
    if (track) {
        s.pending = true;
        s.pend_faces = num_faces;
        s.pend_size = image_size;
    }
    return NR_OK;
}

int nr_compute_weight_map(const float *faces, const int32_t *face_index_map, float *weight_map,
                          int32_t batch, int32_t num_faces, int32_t image_size, void *stream_) {
    if (!faces || !face_index_map || !weight_map) return fail(NR_ERR_INVALID_ARGUMENT, "NULL pointer");
    if (batch < 0 || num_faces < 0 || image_size <= 0) return fail(NR_ERR_INVALID_ARGUMENT, "bad extents");
    cudaError_t e = nr::launch_weight_map_compat(faces, face_index_map, weight_map, batch, num_faces,
                                                 image_size, (cudaStream_t)stream_);
    if (e != cudaSuccess) return fail_cuda(e, "compute_weight_map");
    return NR_OK;
}

}  // extern "C"
