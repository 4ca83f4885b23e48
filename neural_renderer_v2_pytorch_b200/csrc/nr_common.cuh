// nr_common.cuh -- shared device code of the B200-native rasterizer.
//
// The z-buffer result must be bit-identical to the reference kernel
// (neural_renderer_torch/cuda/rasterize_cuda_kernel.cu:52-153), whose SASS contracts some
// products into FMAs and not others.  Everything that decides coverage or depth is therefore
// spelled with explicit rounding intrinsics (never re-contracted by nvcc); the formulas are the
// ones in oracle/nr_oracle.c, which cites the reference line by line.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace nr {

constexpr int TILE = 16;            // tile edge in pixels (internal resolution)
constexpr int TILE_THREADS = 256;   // one thread per pixel of a tile
constexpr int WARP_BW = 8;          // a warp's 8 x 4 pixel block in tile_pixel() and shade_block()
constexpr int WARP_BH = 4;

// nrRasterConfig.flags (include/nr_b200.h)
constexpr int FLAG_RGB = 1, FLAG_SIL = 2, FLAG_DEPTH = 4, FLAG_BACKSIDE = 8, FLAG_AA = 16,
              FLAG_DETERMINISTIC = 32;
// Dense meshes (hundreds of faces per 16x16 tile) are binned into 8x8 tiles instead: four times shorter
// lists to sort and to walk (general binning path and the FINE raster variants only).
constexpr int FINE_TILE = 8;

// Workspace header (device side). Layout shared by all kernels.
struct BinHeader {
    int total_pairs;
    int max_tile_faces;
    int overflow;
    int bad_index;
    int work_counter;   // dynamic tile scheduler of the persistent raster kernel
    // z-buffer path (nr_raster_zbuf.cu)
    int zb_big;         // faces queued for the warp-per-face pass
    int zb_slots;       // contested pixels
    int zb_nodes;       // candidates collected for them
    int zb_work[4];     // dynamic schedulers of its persistent kernels
    int pad[52];
};

// Non-empty tiles of one forward call, consumed by the raster kernel and again by the backward.
// The tiles are kept in TILE_CLASSES regions by list length, longest lists first, so that the
// dynamically scheduled raster kernel starts with the expensive tiles and ends with cheap ones:
//   list[k], k < TILE_CLASSES = number of entries of class k
//   entry i of class k = 4 ints at list[TILE_LIST_HDR + 4 (k cap + i)], cap = views * tiles_per_view:
//   (view, tile_x | tile_y << 16, offset of the tile's face list in the pair array, its length)
constexpr int TILE_LIST_HDR = 8;
constexpr int TILE_ENTRY_INTS = 4;
constexpr int TILE_CLASSES = 4;
__host__ __device__ inline int tile_class(int n) { return n > 96 ? 0 : (n > 48 ? 1 : (n > 24 ? 2 : 3)); }

struct TileList {
    const int4 *entries;
    int cap, total;
    int c[TILE_CLASSES];
};
__device__ __forceinline__ TileList open_tile_list(const int32_t *list, int cap) {
    TileList t;
    t.entries = reinterpret_cast<const int4 *>(list + TILE_LIST_HDR);
    t.cap = cap;
    t.total = 0;
#pragma unroll
    for (int k = 0; k < TILE_CLASSES; ++k) {
        t.c[k] = list[k];
        t.total += t.c[k];
    }
    return t;
}
// i-th tile in heavy-first order
__device__ __forceinline__ int4 tile_entry(const TileList &t, int i) {
    int k = 0;
#pragma unroll
    for (int j = 0; j < TILE_CLASSES - 1; ++j)
        if (k == j && i >= t.c[j]) {
            i -= t.c[j];
            ++k;
        }
    return __ldg(t.entries + (size_t)k * t.cap + i);
}
static_assert(sizeof(BinHeader) == 256, "header is one 256-byte block");

// Per (view, face) record written by the setup kernel: 48 bytes, three float4 loads.
//   q0 = x0 y0 z0 x1 | q1 = y1 z1 x2 y2 | q2 = z2, bbox_x (lo | hi << 16), bbox_y, unused
// A dead face (culled, degenerate, non-finite or off-screen) has bbox_x = 0x0000ffff (lo > hi).
struct FaceRec {
    float4 q0, q1, q2;
};
constexpr uint32_t DEAD_BBOX = 0x0000ffffu;

__device__ __forceinline__ float pix_center(int i, int R) {
    // rasterize_cuda_kernel.cu:76-77: (2.*i + 1 - is) / is evaluated in double then narrowed;
    // numerator and denominator are exact small integers so this is one IEEE float division.
    return __fdiv_rn((float)(2 * i + 1 - R), (float)R);
}

// Pixel-centre coordinates of one resolution.  For a power-of-two R the division is an exact scaling,
// so a multiplication by 1/R gives the same bits as the reference's division.
struct PixGrid {
    int R;
    float invR;
    bool pow2;
    __device__ __forceinline__ explicit PixGrid(int R_) : R(R_), invR(1.f / (float)R_), pow2((R_ & (R_ - 1)) == 0) {}
    __device__ __forceinline__ float center(int i) const {
        return pow2 ? __fmul_rn((float)(2 * i + 1 - R), invR) : pix_center(i, R);
    }
};

// smallest i in [0, R] with center(i) >= v   (R if none).  The float guess is only a starting point:
// the two loops make the result exact for any guess (center() is strictly increasing in i).
__device__ __forceinline__ int first_pixel_ge(float v, const PixGrid &g) {
    const int R = g.R;
    if (g.pow2) {
        // center(i) = (2i + 1 - R) / R exactly, and t = v * R is exact too: center(i) >= v  <=>  2i + 1 - R >= ceil(t)
        const float t = fminf(fmaxf(__fmul_rn(v, (float)R), -2.f * (float)R), 2.f * (float)R);
        return min(max((__float2int_ru(t) + R) >> 1, 0), R);
    }
    const float t = fmaf(v, 0.5f * (float)R, 0.5f * (float)(R - 1));
    int i = (t > 0.f) ? ((t >= (float)R) ? R : (int)ceilf(t)) : 0;      // NaN -> 0
    while (i > 0 && g.center(i - 1) >= v) --i;
    while (i < R && g.center(i) < v) ++i;
    return i;
}

// largest i in [-1, R-1] with center(i) <= v   (-1 if none)
__device__ __forceinline__ int last_pixel_le(float v, const PixGrid &g) {
    const int R = g.R;
    if (g.pow2) {
        // center(i) <= v  <=>  2i + 1 - R <= floor(t)
        const float t = fminf(fmaxf(__fmul_rn(v, (float)R), -2.f * (float)R), 2.f * (float)R);
        return min(max((__float2int_rd(t) + R - 1) >> 1, -1), R - 1);
    }
    const float t = fmaf(v, 0.5f * (float)R, 0.5f * (float)(R - 1));
    int i = (t >= 0.f) ? ((t >= (float)(R - 1)) ? R - 1 : (int)floorf(t)) : -1;   // NaN -> -1
    while (i < R - 1 && g.center(i + 1) <= v) ++i;
    while (i >= 0 && g.center(i) > v) --i;
    return i;
}

// Record of face f of one view (vb = that view's vertices, faces = its face rows) and its exact pixel box; returns false for
// a face no pixel can accept (its record then carries the dead box).
__device__ __forceinline__ bool make_face_record(const float *__restrict__ vb, const int32_t *__restrict__ faces,
                                                 int f, int nv, int R, int draw_backside, FaceRec &r, int &xlo,
                                                 int &xhi, int &ylo, int &yhi, BinHeader *__restrict__ hdr) {
    int i0, i1, i2;
    if (faces) {
        i0 = __ldg(faces + 3 * f + 0);
        i1 = __ldg(faces + 3 * f + 1);
        i2 = __ldg(faces + 3 * f + 2);
    } else {
        i0 = 3 * f;
        i1 = i0 + 1;
        i2 = i0 + 2;
    }
    r.q0 = make_float4(0.f, 0.f, 0.f, 0.f);
    r.q1 = r.q0;
    r.q2 = make_float4(0.f, __uint_as_float(DEAD_BBOX), 0.f, 0.f);
    if ((unsigned)i0 >= (unsigned)nv || (unsigned)i1 >= (unsigned)nv || (unsigned)i2 >= (unsigned)nv) {
        atomicOr(&hdr->bad_index, 1);
        return false;
    }
    const float x0 = vb[3 * i0], y0 = vb[3 * i0 + 1], z0 = vb[3 * i0 + 2];
    const float x1 = vb[3 * i1], y1 = vb[3 * i1 + 1], z1 = vb[3 * i1 + 2];
    const float x2 = vb[3 * i2], y2 = vb[3 * i2 + 1], z2 = vb[3 * i2 + 2];
    r.q0 = make_float4(x0, y0, z0, x1);
    r.q1 = make_float4(y1, z1, x2, y2);
    r.q2.x = z2;

    // A face with a non-finite x or y can never win a pixel in the reference: its barycentric
    // weights divide inf by inf (NaN depth), and NaN fails the z-test (DESIGN.md "Dropped faces").
    bool alive = isfinite(x0) && isfinite(x1) && isfinite(x2) && isfinite(y0) && isfinite(y1) &&
                 isfinite(y2);
    // rasterize_cuda_kernel.cu:100-104, two rounded products
    if (alive && !draw_backside) {
        const float a = __fmul_rn(__fsub_rn(y2, y0), __fsub_rn(x1, x0));
        const float c = __fmul_rn(__fsub_rn(y1, y0), __fsub_rn(x2, x0));
        if (a > c) alive = false;
    }
    // :118-121
    if (alive) {
        const float det = __fmaf_rn(x1, __fsub_rn(y2, y0),
                                    __fmaf_rn(x2, __fsub_rn(y0, y1), __fmul_rn(x0, __fsub_rn(y1, y2))));
        if ((double)fabsf(det) < 0.00000001) alive = false;
    }
    xlo = 1; xhi = 0; ylo = 1; yhi = 0;
    if (alive) {
        // :94-97  pixel passes iff  min <= centre <= max  on both axes
        const PixGrid grid(R);
        xlo = first_pixel_ge(fminf(x0, fminf(x1, x2)), grid);
        xhi = last_pixel_le(fmaxf(x0, fmaxf(x1, x2)), grid);
        ylo = first_pixel_ge(fminf(y0, fminf(y1, y2)), grid);
        yhi = last_pixel_le(fmaxf(y0, fmaxf(y1, y2)), grid);
        if (xlo > xhi || ylo > yhi) alive = false;
    }
    if (alive) {
        r.q2.y = __uint_as_float((uint32_t)xlo | ((uint32_t)xhi << 16));
        r.q2.z = __uint_as_float((uint32_t)ylo | ((uint32_t)yhi << 16));
    }
    return alive;
}

// Raw (un-normalised) barycentric numerators, rasterize_cuda_kernel.cu:130-132 / :276-278.
__device__ __forceinline__ void raw_weights(float xp, float yp, float x0, float y0, float x1,
                                            float y1, float x2, float y2, float &w0, float &w1,
                                            float &w2) {
    w0 = __fadd_rn(__fmaf_rn(yp, __fsub_rn(x2, x1), __fmul_rn(xp, __fsub_rn(y1, y2))),
                   __fmaf_rn(x1, y2, -__fmul_rn(x2, y1)));
    w1 = __fadd_rn(__fmaf_rn(yp, __fsub_rn(x0, x2), __fmul_rn(xp, __fsub_rn(y2, y0))),
                   __fmaf_rn(x2, y0, -__fmul_rn(x0, y2)));
    w2 = __fadd_rn(__fmaf_rn(yp, __fsub_rn(x1, x0), __fmul_rn(xp, __fsub_rn(y0, y1))),
                   __fmaf_rn(x0, y1, -__fmul_rn(x1, y0)));
}

// IEEE division where a result must be bit-identical to the reference (everything the FORWARD
// writes); the backward only needs its gradients to ~1e-6 relative and may use the fast one.
template <bool EXACT>
__device__ __forceinline__ float div_f(float a, float b) {
    return EXACT ? __fdiv_rn(a, b) : __fdividef(a, b);
}

// compute_weight_map_cuda_kernel, rasterize_cuda_kernel.cu:279-306, from the raw numerators.
template <bool EXACT = true>
__device__ __forceinline__ void normalize_weights(float &w0, float &w1, float &w2) {
    if (__fadd_rn(__fadd_rn(w0, w1), w2) < 0.f) {
        w0 = -w0;
        w1 = -w1;
        w2 = -w2;
    }
    w0 = fmaxf(w0, 0.f);
    w1 = fmaxf(w1, 0.f);
    w2 = fmaxf(w2, 0.f);
    const float s = __fadd_rn(__fadd_rn(w0, w1), w2);
    w0 = fmaxf(fminf(div_f<EXACT>(w0, s), 1.f), 0.f);
    w1 = fmaxf(fminf(div_f<EXACT>(w1, s), 1.f), 0.f);
    w2 = fmaxf(fminf(div_f<EXACT>(w2, s), 1.f), 0.f);
}

// utils.maximum (utils.py:91-101) on scalars.
__device__ __forceinline__ float nr_maximum(float r, float l) {
    if (fmaxf(r, l) <= 0.f) return 0.f;
    if (fabsf(__fsub_rn(r, l)) < 1e-4f) return 0.f;
    return (r > l) ? -r : l;
}

// Perspective-correct texel coordinate of a foreground pixel, rasterize.py:111-121, with every
// operation rounded separately like the chain of torch ops it restates.  Forward and backward both
// call this, so they agree on which four texels a pixel touches.
struct TexCoord {
    float depth, nx, ny;   // 1 / sum(w/z'), sum(w u / z'), sum(w v / z')
    float x0, y0;          // before the clamp
    float xf, yf;          // after the clamp to [min corner, max corner - eps]
    float zz[3];           // z + 1e-10
};
template <bool EXACT = true>
__device__ __forceinline__ TexCoord texel_coord(const float q[3], const float z[3], const float u[3],
                                                const float v[3], float eps) {
    TexCoord t;
    t.zz[0] = __fadd_rn(z[0], 1e-10f);
    t.zz[1] = __fadd_rn(z[1], 1e-10f);
    t.zz[2] = __fadd_rn(z[2], 1e-10f);
    const float a0 = __fadd_rn(div_f<EXACT>(q[0], t.zz[0]), 1e-10f);
    const float a1 = __fadd_rn(div_f<EXACT>(q[1], t.zz[1]), 1e-10f);
    const float a2 = __fadd_rn(div_f<EXACT>(q[2], t.zz[2]), 1e-10f);
    t.depth = div_f<EXACT>(1.f, __fadd_rn(__fadd_rn(a0, a1), a2));
    t.nx = __fadd_rn(__fadd_rn(div_f<EXACT>(__fmul_rn(q[0], u[0]), t.zz[0]), div_f<EXACT>(__fmul_rn(q[1], u[1]), t.zz[1])),
                     div_f<EXACT>(__fmul_rn(q[2], u[2]), t.zz[2]));
    t.ny = __fadd_rn(__fadd_rn(div_f<EXACT>(__fmul_rn(q[0], v[0]), t.zz[0]), div_f<EXACT>(__fmul_rn(q[1], v[1]), t.zz[1])),
                     div_f<EXACT>(__fmul_rn(q[2], v[2]), t.zz[2]));
    t.x0 = __fmul_rn(t.nx, t.depth);
    t.y0 = __fmul_rn(t.ny, t.depth);
    t.xf = fminf(fmaxf(t.x0, fminf(u[0], fminf(u[1], u[2]))), __fsub_rn(fmaxf(u[0], fmaxf(u[1], u[2])), eps));
    t.yf = fminf(fmaxf(t.y0, fminf(v[0], fminf(v[1], v[2]))), __fsub_rn(fmaxf(v[0], fmaxf(v[1], v[2])), eps));
    return t;
}

// The same from the three quotients the forward stored (aux_map): no division left.
__device__ __forceinline__ TexCoord texel_coord_stored(float depth, float nx, float ny, const float z[3], const float u[3],
                                                       const float v[3], float eps) {
    TexCoord t;
    t.zz[0] = __fadd_rn(z[0], 1e-10f);
    t.zz[1] = __fadd_rn(z[1], 1e-10f);
    t.zz[2] = __fadd_rn(z[2], 1e-10f);
    t.depth = depth;
    t.nx = nx;
    t.ny = ny;
    t.x0 = __fmul_rn(nx, depth);
    t.y0 = __fmul_rn(ny, depth);
    t.xf = fminf(fmaxf(t.x0, fminf(u[0], fminf(u[1], u[2]))), __fsub_rn(fmaxf(u[0], fmaxf(u[1], u[2])), eps));
    t.yf = fminf(fmaxf(t.y0, fminf(v[0], fminf(v[1], v[2]))), __fsub_rn(fmaxf(v[0], fmaxf(v[1], v[2])), eps));
    return t;
}

// Lights as the kernels see them (include/nr_b200.h: nrLights).
struct LightArgs {
    int num;
    const int32_t *types;
    const float *data;       // [L, B, 8]
    const float *vnormals;   // [B, nv, 3]
    float *grad_vnormals;    // backward
    const float *backgrounds;   // [B, 3, R, R] output orientation, or null
};

// Colour weight of one pixel from its interpolated normal n (rasterize.py:256-282), and when
// gn != nullptr the gradient of  sum_c gcw[c] * cw[c]  with respect to n.
__device__ __forceinline__ void light_weights(const LightArgs &L, int b, int B, const float n[3], float cw[3],
                                              const float *gcw, float *gn) {
    cw[0] = cw[1] = cw[2] = 0.f;
    if (gn) gn[0] = gn[1] = gn[2] = 0.f;
    for (int l = 0; l < L.num; ++l) {
        const int type = __ldg(L.types + l);
        const float *d = L.data + ((size_t)l * B + b) * 8;
        const float cr = __ldg(d), cg = __ldg(d + 1), cb = __ldg(d + 2);
        const int kind = type & 3;
        if (kind == 0) {
            cw[0] = __fadd_rn(cw[0], cr); cw[1] = __fadd_rn(cw[1], cg); cw[2] = __fadd_rn(cw[2], cb);
            continue;
        }
        float dir[3] = {0.f, 0.f, 1.f};                     // specular: direction_eye (rasterize.py:271)
        if (kind == 1) { dir[0] = __ldg(d + 3); dir[1] = __ldg(d + 4); dir[2] = __ldg(d + 5); }
        const float raw = __fadd_rn(__fadd_rn(__fmul_rn(-dir[0], n[0]), __fmul_rn(-dir[1], n[1])), __fmul_rn(-dir[2], n[2]));
        const bool backside = (type & 4) != 0;
        const float a = backside ? fabsf(raw) : fmaxf(raw, 0.f);
        const float gate = backside ? (raw > 0.f ? 1.f : (raw < 0.f ? -1.f : 0.f)) : (raw > 0.f ? 1.f : 0.f);
        float inten = a, dinten = gate;                     // d inten / d raw
        if (kind == 2) {
            const float alpha = __ldg(d + 6);
            inten = powf(a, alpha);
            dinten = gate * alpha * powf(a, alpha - 1.f);
            if (gate == 0.f) dinten = 0.f;
        }
        cw[0] = __fadd_rn(cw[0], __fmul_rn(inten, cr));
        cw[1] = __fadd_rn(cw[1], __fmul_rn(inten, cg));
        cw[2] = __fadd_rn(cw[2], __fmul_rn(inten, cb));
        if (gn) {
            const float gi = (gcw[0] * cr + gcw[1] * cg + gcw[2] * cb) * dinten;
            gn[0] -= gi * dir[0]; gn[1] -= gi * dir[1]; gn[2] -= gi * dir[2];
        }
    }
}

// Thread -> pixel mapping inside a tile: warp w owns the 8x4 block at
// ((w & 1) * 8, (w >> 1) * 4); lane l is pixel (l & 7, l >> 3) of the block.
__device__ __forceinline__ void tile_pixel(int tid, int &px, int &py) {
    const int w = tid >> 5, l = tid & 31;
    px = (w & 1) * WARP_BW + (l & 7);
    py = (w >> 1) * WARP_BH + (l >> 3);
}

}  // namespace nr
