// nr_shade.cuh -- device code shared by the two raster kernels (nr_raster.cu: one warp per 8x8 pixel block
// walking sorted tile lists; nr_raster_dense.cu: one CTA per tile, one thread per face, for meshes of small
// triangles): the reference's depth arithmetic, the output fills and the fused shading epilogue.
#pragma once
#include "nr_kernels.h"

namespace nr {

// ---- depth of a pixel inside a face --------------------------------------------------------------------
// rasterize_cuda_kernel.cu:129-139, bit for bit (SURVEY.md 2.3): normalised weights by IEEE divisions,
// zp = rcp_rn(w0/z0 + w1/z1 + w2/z2).  w0..w2 are the raw numerators of raw_weights().
__device__ __forceinline__ float exact_zp(float w0, float w1, float w2, float z0, float z1, float z2) {
    const float ws = __fadd_rn(__fadd_rn(w0, w1), w2);
    const float n0 = __fdiv_rn(w0, ws), n1 = __fdiv_rn(w1, ws), n2 = __fdiv_rn(w2, ws);
    const float s = __fadd_rn(__fadd_rn(__fdiv_rn(n0, z0), __fdiv_rn(n1, z1)), __fdiv_rn(n2, z2));
    return __frcp_rn(s);
}

// The same depth with four roundings less and no IEEE division: zp ~ ws / (w0/z0 + w1/z1 + w2/z2) with the
// reciprocals iz_k = rcp_rn(z_k) taken once per face.  Only trusted for REGULAR candidates: all three weights
// of one sign (zeros allowed) and all three depths positive and of ordinary magnitude (face_z_regular), so
// that nothing cancels: then both this value and exact_zp() are within a few ulp of the real-number depth,
// |fast - exact| <= 12 ulp < FAST_Z_REL * zp, and the depth lies in [min z, max z] up to that error.
constexpr float FAST_Z_REL = 2e-6f;
__device__ __forceinline__ bool face_z_regular(float z0, float z1, float z2) {
    return z0 > 1e-18f && z1 > 1e-18f && z2 > 1e-18f && z0 < 1e18f && z1 < 1e18f && z2 < 1e18f;   // NaN fails
}
__device__ __forceinline__ bool weights_one_sign(float w0, float w1, float w2) {
    return (w0 >= 0.f && w1 >= 0.f && w2 >= 0.f) || (w0 <= 0.f && w1 <= 0.f && w2 <= 0.f);         // NaN fails
}
__device__ __forceinline__ float fast_rcp(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float fast_zp(float w0, float w1, float w2, float iz0, float iz1, float iz2) {
    const float ws = (w0 + w1) + w2;
    return __fdividef(ws, fmaf(w0, iz0, fmaf(w1, iz1, w2 * iz2)));
}

// Perspective-correct bilinear texture sample of one foreground pixel, rasterize.py:100-153.
// q = weight map, z = face depths, uv = texel coordinates of the 3 face corners.
__device__ __forceinline__ void sample_texture(const float *__restrict__ tex_b, int H, int W,
                                               float eps, const float q[3], const float z[3],
                                               const float u[3], const float v[3], float rgb[3], TexCoord &tc) {
    tc = texel_coord(q, z, u, v, eps);
    const float xf = tc.xf, yf = tc.yf;
    const float xff = floorf(xf), yff = floorf(yf);
    const float xcf = __fadd_rn(xff, 1.f), ycf = __fadd_rn(yff, 1.f);
    const int xfi = (int)xff, yfi = (int)yff, xci = (int)xcf, yci = (int)ycf;
    const float w1 = __fmul_rn(__fsub_rn(ycf, yf), __fsub_rn(xcf, xf));
    const float w2 = __fmul_rn(__fsub_rn(ycf, yf), __fsub_rn(xf, xff));
    const float w3 = __fmul_rn(__fsub_rn(yf, yff), __fsub_rn(xcf, xf));
    const float w4 = __fmul_rn(__fsub_rn(yf, yff), __fsub_rn(xf, xff));
    const int T = H * W;
    const int i1 = yfi * W + xfi, i2 = yfi * W + xci, i3 = yci * W + xfi, i4 = yci * W + xci;
    // to_map (utils.py:104-114) yields zero for a negative index; an index >= H*W is an
    // IndexError in the reference and reads as zero here.
    const bool ok1 = (unsigned)i1 < (unsigned)T, ok2 = (unsigned)i2 < (unsigned)T;
    const bool ok3 = (unsigned)i3 < (unsigned)T, ok4 = (unsigned)i4 < (unsigned)T;
    const float *p1 = tex_b + i1, *p2 = tex_b + i2, *p3 = tex_b + i3, *p4 = tex_b + i4;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int o = c * T;
        const float t1 = ok1 ? __ldg(p1 + o) : 0.f, t2 = ok2 ? __ldg(p2 + o) : 0.f;
        const float t3 = ok3 ? __ldg(p3 + o) : 0.f, t4 = ok4 ? __ldg(p4 + o) : 0.f;
        rgb[c] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w1, t1), __fmul_rn(w2, t2)), __fmul_rn(w3, t3)),
                           __fmul_rn(w4, t4));
    }
}

// ---- output initialisation, done by the raster kernel itself --------------------------------------
// The raster kernel is instruction-issue bound and leaves HBM idle, so everything that is a plain
// fill rides along in it instead of running in front of it: the pixels of EMPTY tiles (face index -1,
// image 0 or the background picture), and the caller's `zero` buffers (the gradient accumulators of the
// coming backward).  Pixels of non-empty tiles are all written by the raster items, foreground or not.

// value of rgb channel c behind a background pixel at OUTPUT position (u, v) of view b
template <bool FULL>
__device__ __forceinline__ float background_value(const RasterArgs &a, int b, int c, int u, int v) {
    if (!FULL || !a.lights.backgrounds || c >= 3 || !(a.flags & FLAG_RGB)) return 0.f;
    return __ldg(a.lights.backgrounds + (((size_t)b * 3 + c) * a.R + u) * a.R + v);
}

// `sparse`: write only what nr_rasterize_backward reads, i.e. not the face index of an empty tile, and
// its internal-resolution image (anti-aliasing) only when a neighbouring tile is non-empty (the stencil
// of a foreground pixel reaches one pixel into the next tile).
template <bool AA, bool FULL, bool FINE>
__device__ __forceinline__ void fill_empty_tile(const RasterArgs &a, int b, int tx, int ty, int lane, bool sparse) {
    const int R = a.R, S = a.S, C = a.C;
    constexpr bool aa = AA;
    constexpr int TSZ = FINE ? FINE_TILE : TILE;
    bool need_fim = true, need_internal = true;
    if (sparse) {
        need_fim = false;
        if (aa) {
            const int *tc = a.tile_count + (size_t)b * a.ntx * a.ntx;
            int any = 0;
            for (int dy = -1; dy <= 1; ++dy)
                for (int dx = -1; dx <= 1; ++dx) {
                    const int x = tx + dx, y = ty + dy;
                    if (x >= 0 && y >= 0 && x < a.ntx && y < a.ntx) any |= __ldg(tc + y * a.ntx + x);
                }
            need_internal = any != 0;
        }
    }
    if (!FINE && (!FULL || ((R & 15) == 0 && !a.lights.backgrounds))) {
        // vector path: a tile row is 64 aligned bytes in every plane; the flipped tile is again a tile
        const int r = lane >> 2, q = (lane & 3) * 4;
        const int4 m1 = make_int4(-1, -1, -1, -1);
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        if (need_fim) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int y = ty * TILE + r + 8 * h;
                __stcs(reinterpret_cast<int4 *>(a.fim + ((size_t)b * R + y) * R + tx * TILE + q), m1);
            }
        }
        if (!a.images) return;
        const int u0 = R - TILE - ty * TILE, v0 = R - TILE - tx * TILE;
        float *full = aa ? a.internal : a.images;          // internal-resolution planes
        if (!aa || need_internal) {
            for (int c = 0; c < C; ++c) {
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    __stcs(reinterpret_cast<float4 *>(full + (((size_t)b * C + c) * R + u0 + r + 8 * h) * R + v0 + q), z);
            }
        }
        if (aa) {
            for (int i = lane; i < C * 16; i += 32) {
                const int c = i >> 4, rr = (i >> 1) & 7, hh = (i & 1) * 4;
                __stcs(reinterpret_cast<float4 *>(a.images + (((size_t)b * C + c) * S + (u0 >> 1) + rr) * S + (v0 >> 1) + hh), z);
            }
        }
        return;
    }
    // (the launcher sends everything the vector path cannot do to the FULL variant)
    if constexpr (FULL) {
    for (int p = lane; p < TSZ * TSZ; p += 32) {
        const int xi = tx * TSZ + (p & (TSZ - 1)), yi = ty * TSZ + p / TSZ;
        if (xi >= R || yi >= R) continue;
        if (need_fim) a.fim[((size_t)b * R + yi) * R + xi] = -1;
        if (!a.images) continue;
        const int u = R - 1 - yi, v = R - 1 - xi;
        float *full = aa ? a.internal : a.images;
        for (int c = 0; c < C; ++c) {
            if (!aa || need_internal) full[(((size_t)b * C + c) * R + u) * R + v] = background_value<FULL>(a, b, c, u, v);
            if (aa && !(u & 1) && !(v & 1)) {
                // rasterize.py:323-328 on a pure-background quad
                const float sum = __fadd_rn(__fadd_rn(__fadd_rn(background_value<FULL>(a, b, c, u, v), background_value<FULL>(a, b, c, u + 1, v)),
                                                      background_value<FULL>(a, b, c, u, v + 1)), background_value<FULL>(a, b, c, u + 1, v + 1));
                a.images[(((size_t)b * C + c) * S + (u >> 1)) * S + (v >> 1)] = __fmul_rn(sum, 0.25f);
            }
        }
    }
}
}

// ---- fill items ------------------------------------------------------------------------------------------
// Work that is stores only, interleaved with the raster items so that it drains to HBM all along the kernel
// instead of in one burst: fill item i < B * tiles is tile i if it is empty; then come 4 KB chunks of the
// caller's zero buffers.  One warp performs one fill item.
constexpr int ZCHUNK = 256;                 // int4 per chunk
struct FillPlan {
    int all_tiles, fill_items;
    int zero_chunks[4];
};
__device__ __forceinline__ FillPlan make_fill_plan(const RasterArgs &a) {
    FillPlan p;
    p.all_tiles = a.B * a.ntx * a.ntx;
    p.fill_items = p.all_tiles;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        p.zero_chunks[k] = 0;
        if (k < a.num_zero) {
            p.zero_chunks[k] = (int)((a.zero_bytes[k] >> 4) / ZCHUNK) + 1;      // the last chunk also takes the tail words
            p.fill_items += p.zero_chunks[k];
        }
    }
    return p;
}
template <bool AA, bool FULL, bool FINE>
__device__ __forceinline__ void do_fill_item(const RasterArgs &a, const FillPlan &p, int i, int lane) {
    if (i < p.all_tiles) {
        if (__ldg(a.tile_count + i) != 0) return;
        const int nt = a.ntx * a.ntx;
        int b, tx, ty;
        if ((a.ntx & (a.ntx - 1)) == 0) {       // power-of-two tile grid: shifts instead of divisions
            const int sh = __ffs(a.ntx) - 1;
            b = i >> (2 * sh);
            ty = (i >> sh) & (a.ntx - 1);
            tx = i & (a.ntx - 1);
        } else {
            b = i / nt;
            const int tt = i - b * nt;
            ty = tt / a.ntx;
            tx = tt - ty * a.ntx;
        }
        fill_empty_tile<AA, FULL, FINE>(a, b, tx, ty, lane, a.sparse_maps != 0);
        return;
    }
    int j = i - p.all_tiles;
    for (int k = 0; k < a.num_zero; ++k) {
        if (j >= p.zero_chunks[k]) {
            j -= p.zero_chunks[k];
            continue;
        }
        int4 *dst = reinterpret_cast<int4 *>(a.zero_ptr[k]);
        const size_t n16 = a.zero_bytes[k] >> 4, base = (size_t)j * ZCHUNK;
#pragma unroll
        for (int s = 0; s < ZCHUNK / 32; ++s) {
            const size_t idx = base + lane + 32 * s;
            if (idx < n16) __stcs(dst + idx, make_int4(0, 0, 0, 0));
        }
        if (j == p.zero_chunks[k] - 1 && lane < (int)((a.zero_bytes[k] & 15) >> 2))
            reinterpret_cast<int32_t *>(dst + n16)[lane] = 0;
        return;
    }
}

// ---- epilogue: every pixel of an 8x4 block is written ------------------------------------------------------
// Called by ALL 32 lanes of a warp whose lane l owns pixel (xi, yi) = block origin + (l & 7, l >> 3) (the
// anti-aliasing mean goes through quad shuffles).  best = winning face or -1, (bw0..2) its raw weight
// numerators at this pixel, (bz0..2) its corner depths.  Fuses rasterize_cuda_kernel.cu:246-308 (weight map),
// rasterize.py:100-153 (texture sampling), :252-283 (lights), :240-242 (silhouettes), :80-88 (depth),
// :295-310 (channel merge), :315-316 (permute + flip), :321-328 (2x2 anti-aliasing mean).
template <bool RGB, bool AA, bool FULL>
__device__ __forceinline__ void shade_block(const RasterArgs &a, int b, int xi, int yi, bool valid, int best,
                                            float bw0, float bw1, float bw2, float bz0, float bz1, float bz2,
                                            bool has_bg) {
    constexpr bool aa = AA;
    const int R = a.R;
    if (__ballot_sync(0xffffffffu, best >= 0) == 0u && !has_bg) {
        // nothing but (black) background in this block
        if (valid) {
            a.fim[((size_t)b * R + yi) * R + xi] = -1;
            if (!FULL || a.images) {
                const int u_ = R - 1 - yi, v_ = R - 1 - xi, C = a.C;
                float *full = (aa ? a.internal : a.images) + ((size_t)b * C * R + u_) * R + v_;
                const int plane = R * R;
                for (int c = 0; c < C; ++c) full[c * plane] = 0.f;
                if (aa && !(xi & 1) && !(yi & 1)) {
                    float *half = a.images + ((size_t)b * C * a.S + (u_ >> 1)) * a.S + (v_ >> 1);
                    const int plane_h = a.S * a.S;
                    for (int c = 0; c < C; ++c) half[c * plane_h] = 0.f;
                }
            }
        }
        return;
    }
    const bool fg = valid && best >= 0;
    float q[3] = {0.f, 0.f, 0.f};
    if (fg) {
        q[0] = bw0; q[1] = bw1; q[2] = bw2;
        normalize_weights(q[0], q[1], q[2]);
    }
    const size_t pix = ((size_t)b * R + yi) * R + xi;
    float dm = 0.f;
    if (valid) a.fim[pix] = fg ? best : -1;
    // forward -> backward state (nr_b200.h: aux_map): the weights here, the texel coordinate below
    float *aux = (fg && a.aux) ? a.aux + pix * (RGB ? 6 : 3) : nullptr;
    if (aux && !RGB) {
        aux[0] = q[0]; aux[1] = q[1]; aux[2] = q[2];
    }
    if (fg) {
        if (FULL && a.wmap) {
            float *w = a.wmap + pix * 3;
            w[0] = q[0]; w[1] = q[1]; w[2] = q[2];
        }
        if ((a.flags & FLAG_DEPTH) || (FULL && a.dmap))
            dm = __fdiv_rn(1.f, __fadd_rn(__fadd_rn(__fdiv_rn(q[0], bz0), __fdiv_rn(q[1], bz1)), __fdiv_rn(q[2], bz2)));
        if (FULL && a.dmap) a.dmap[pix] = dm;
    }
    if (!FULL || a.images) {
        const int C = a.C, S = a.S;
        const int u_ = R - 1 - yi, v_ = R - 1 - xi;   // flipped coordinates, rasterize.py:316
        // one 64-bit pointer per output (this pixel, channel 0); channel c is a 32-bit plane offset away
        float *p_full = (aa ? a.internal : a.images) + ((size_t)b * C * R + u_) * R + v_;
        float *p_half = aa ? a.images + ((size_t)b * C * S + (u_ >> 1)) * S + (v_ >> 1) : nullptr;
        const int plane_full = R * R, plane_half = S * S;
        // one channel value of this pixel -> images (and the internal-resolution copy under AA)
        auto put = [&](int c, float val) {
            // background pixels show the background picture (black without one)
            if (has_bg && !fg && valid) val = background_value<FULL>(a, b, c, u_, v_);
            if (valid) p_full[c * plane_full] = val;
            if (!aa) return;
            // quad in flipped coordinates: F[2Y][2X] is (yi odd, xi odd); rasterize.py:323-328
            const float px_ = __shfl_xor_sync(0xffffffffu, val, 1);   // same row, other column
            const float py_ = __shfl_xor_sync(0xffffffffu, val, 8);   // other row, same column
            const float pd_ = __shfl_xor_sync(0xffffffffu, val, 9);
            if (valid && !(xi & 1) && !(yi & 1)) {
                // me = (even, even) -> F[2Y+1][2X+1]; py_ = (odd row, even col) -> F[2Y][2X+1]
                // px_ = (even row, odd col) -> F[2Y+1][2X]; pd_ = (odd, odd) -> F[2Y][2X]
                const float sum = __fadd_rn(__fadd_rn(__fadd_rn(pd_, px_), py_), val);
                p_half[c * plane_half] = __fmul_rn(sum, 0.25f);
            }
        };
        int c = 0;
        if (RGB) {
            float rgb[3] = {0.f, 0.f, 0.f};
            if (fg) {
                const int32_t *fti = a.ft + 3 * (size_t)best;
                const float *vtb = a.vt + (size_t)b * a.nvt * 2;
                float u[3], v[3];
                // a texture-vertex index outside [0, nvt) (an IndexError in the reference, rasterize.py:246)
                // reads nothing: the pixel stays black and the call is flagged (nrBinStats.bad_index & 2)
                bool tex_ok = true;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const int t = __ldg(fti + k);
                    const bool ok = (unsigned)t < (unsigned)a.nvt;
                    tex_ok &= ok;
                    const float2 uv = __ldg(reinterpret_cast<const float2 *>(vtb) + (ok ? t : 0));
                    u[k] = uv.x;
                    v[k] = uv.y;
                }
                const float z[3] = {bz0, bz1, bz2};
                TexCoord tc;
                tc.depth = tc.nx = tc.ny = 0.f;
                if (tex_ok) sample_texture(a.tex + (size_t)b * 3 * a.H * a.W, a.H, a.W, a.eps, q, z, u, v, rgb, tc);
                else atomicOr(&a.hdr->bad_index, 2);
                if (aux) {
                    reinterpret_cast<float2 *>(aux)[0] = make_float2(q[0], q[1]);
                    reinterpret_cast<float2 *>(aux)[1] = make_float2(q[2], tc.depth);
                    reinterpret_cast<float2 *>(aux)[2] = make_float2(tc.nx, tc.ny);
                }
                if (FULL && a.lights.num > 0) {
                    // smooth normal map (rasterize.py:186-187) and light accumulation (:252-283)
                    float n[3] = {0.f, 0.f, 0.f}, cw[3];
                    const float *vnb = a.lights.vnormals + (size_t)b * a.nv * 3;
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        const int vid = a.faces ? __ldg(a.faces + 3 * (size_t)best + k) : 3 * best + k;
#pragma unroll
                        for (int c2 = 0; c2 < 3; ++c2) n[c2] = __fadd_rn(n[c2], __fmul_rn(q[k], __ldg(vnb + 3 * (size_t)vid + c2)));
                    }
                    light_weights(a.lights, b, a.B, n, cw, nullptr, nullptr);
                    rgb[0] = __fmul_rn(rgb[0], cw[0]); rgb[1] = __fmul_rn(rgb[1], cw[1]); rgb[2] = __fmul_rn(rgb[2], cw[2]);
                }
            }
            put(0, rgb[0]);
            put(1, rgb[1]);
            put(2, rgb[2]);
            c = 3;
        }
        if (a.flags & FLAG_SIL) put(c++, fg ? 1.f : 0.f);
        if (a.flags & FLAG_DEPTH) put(c++, dm);
    }
}

}  // namespace nr
