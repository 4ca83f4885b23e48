// nr_kernels.h -- internal launcher interfaces (not part of the C ABI).
#pragma once
#include <cuda.h>       // CUtensorMap (types only: the encoder is fetched through the runtime, no -lcuda)
#include "nr_common.cuh"

namespace nr {

// Tile lists up to this many faces are sorted in shared memory (k_sort_tiles);
// longer ones by k_sort_long in global memory.
constexpr int SMEM_SORT_CAP = 8192;

// Brackets one launch with CUDA events while nr_profile_enable(1) is in force (nr_profile.cu).
enum ProfSlot { PROF_MEMSET = 0, PROF_SETUP, PROF_SCAN, PROF_SCATTER, PROF_SORT_LONG, PROF_RASTER,
                PROF_BACKWARD, PROF_DIFF_BACKWARD, PROF_WEIGHT_MAP, PROF_ZB_FACES, PROF_CAMERA_FORWARD,
                PROF_CAMERA_BACKWARD, PROF_ZB_RESOLVE, PROF_ZB_SHADE };
class ProfScope {
public:
    ProfScope(int slot, cudaStream_t stream);
    ~ProfScope();
private:
    int slot_;
    cudaStream_t stream_;
    void *start_;
};

struct BinningArgs {
    const float *verts;
    const int32_t *faces;   // may be null: face f = vertices 3f..3f+2
    int B, nv, nf, R, draw_backside, ntx;
    FaceRec *rec;
    int *tile_count, *tile_offset, *tile_cursor;
    int32_t *pairs;
    long long pair_capacity;
    BinHeader *hdr;
    int32_t *tile_list;     // [TILE_LIST_HDR + 4 * TILE_CLASSES * B * ntx * ntx] ints, header zeroed here
    int sm_count;
    int one_cta_per_view;   // allow the single-kernel small-mesh path (k_bin_view)
    int tile_shift;         // log2 of the tile edge: 4 (16x16), or 3 (8x8, general path only); ntx counts these tiles
};
bool binning_fits_one_cta_per_view(int nf, int R);
cudaError_t launch_binning(const BinningArgs &a, cudaStream_t stream);

struct RasterArgs {
    const FaceRec *rec;
    const int *tile_count, *tile_offset;
    const int32_t *pairs;
    BinHeader *hdr;
    const int32_t *tile_list;
    int sm_count;
    int B, nf, R, S, ntx, C, flags;
    float near_plane, far_plane, eps, delta;
    const float *vt;        // [B, nvt, 2]
    const int32_t *ft;      // [nf, 3]
    const float *tex;       // [B, 3, H, W]
    int nvt, H, W;
    int32_t *fim;           // [B, R, R]
    float *wmap;            // [B, R, R, 3] or null
    float *dmap;            // [B, R, R] or null
    float *images;          // [B, C, S, S] or null (compat call renders no image)
    float *internal;        // [B, C, R, R] (AA) or null
    float *aux;             // [B, R, R, 6 (rgb) or 3] forward -> backward state at foreground pixels, or null
    const int32_t *faces;   // [nf, 3] vertex ids (null: 3f..3f+2), only read when lights are on
    int nv;
    LightArgs lights;
    int fine;               // 8x8 tiles (ntx and the tile list are in those units)
    int sparse_maps;        // fim / internal only where the backward reads them (see NR_SPARSE_MAPS)
    // z-buffer path for meshes of small triangles (nr_raster_zbuf.cu); null / 0 otherwise
    const float *verts;             // [B, nv, 3]
    unsigned long long *zbuf;       // [B, R, R]  (bits of the cheap depth) << 32 | face
    unsigned *zb_bitmap;            // [B, R, zb_wpr] contested pixels, right behind the header
    unsigned *zb_coarse;            // [B, zb_crows, zb_wpr] OR of eight rows of it, right behind the bitmap
    uint2 *zb_box;                  // [B, nf] exact pixel box of every face (x lo | hi << 16, y lo | hi << 16)
    int zb_wpr, zb_crows;           // 32-bit words per row; ceil(R / 8)
    int *zb_head, *zb_pix_of;       // [zb_slot_cap] candidate list head / pixel of every contested pixel
    int4 *zb_nodes;                 // [zb_node_cap] (face, depth, min corner depth, next)
    int zb_slot_cap, zb_node_cap;
    // buffers the raster kernel zero-fills on the side (16-byte aligned, bytes a multiple of 4)
    int num_zero;
    void *zero_ptr[4];
    size_t zero_bytes[4];
};
cudaError_t launch_background_fill(const RasterArgs &a, cudaStream_t stream);
cudaError_t launch_raster(const RasterArgs &a, cudaStream_t stream);
cudaError_t launch_raster_zbuf(const RasterArgs &a, cudaStream_t stream);      // nr_raster_zbuf.cu

struct BackwardArgs {
    const float *verts;     // [B, nv, 3]
    const int32_t *faces;   // [nf, 3] or null
    const float *vt;
    const int32_t *ft;
    const float *tex;
    const int32_t *fim;
    const float *internal;  // [B, C, R, R] flipped planar
    const float *aux;       // the forward's aux map, or null (weights and texel coordinates are then recomputed)
    const float *grad_images;   // [B, C, S, S]
    const int32_t *tile_list;   // non-empty tiles of the forward, or null (all tiles)
    int sm_count;
    float *grad_verts, *grad_tex, *grad_vt;
    // deterministic mode: 64-bit fixed-point accumulators (same shapes as the three gradients,
    // laid out back to back) and the power-of-two scale; null = float atomics
    long long *det_verts, *det_tex, *det_vt, *det_vn;   // det_vn: grad_vertex_normals (lights)
    float det_scale;
    LightArgs lights;
    int B, nv, nf, R, S, ntx, C, flags, nvt, H, W;
    float eps;
    // gradient of the light data [L, B, 8] (colour 0..2, direction 3..5, alpha 6), accumulated; null = none.
    // Read by the lit variants only.  det_light: its fixed-point accumulator in deterministic mode.
    float *grad_light;
    long long *det_light;
    // Tensor maps of the staged front of k_backward (nr_backward.cu): face_index_map [B, R, R], the stencil image
    // [B*C, R, R] and grad_images [B*C, S, S].  Filled by launch_backward; unused by the unstaged path.
    CUtensorMap map_fim, map_img, map_grad;
};
cudaError_t launch_backward(const BackwardArgs &a, cudaStream_t stream);

// ---- programmatic dependent launch: a kernel launched with launch_after() may start (block scheduling, its
// prologue) while the kernel in front of it on the stream is still draining; it must call pdl_wait() before it
// touches anything that kernel (or an earlier one) wrote, and the kernel in front lets it go with pdl_trigger().
// Both are no-ops in a kernel launched the ordinary way.  It pays where a chain of short kernels is bound by
// launch latency (config 3: -6 %) and costs about 1 % where the kernels fill the machine for long (configs 2 and 4):
// the launchers ask for it for calls of up to PDL_MAX_PIXELS pixels.  NR_PDL=<mask> overrides (0 = never).
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
constexpr long long PDL_MAX_PIXELS = 4ll << 20;
bool pdl_enabled(int which, long long pixels);    // which: 1 raster kernel, 2 backward kernel, 4 passes of the z-buffer path
template <typename... KArgs, typename... Args>
inline cudaError_t launch_after(int which, long long pixels, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled(which, pixels) ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

cudaError_t launch_differentiation_backward(const float *images, const float *grad_output,
                                            float *grad_coordinates, int B, int R, int C,
                                            cudaStream_t stream);

cudaError_t launch_weight_map_compat(const float *faces, const int32_t *fim, float *wmap, int B,
                                     int nf, int R, cudaStream_t stream);

}  // namespace nr
