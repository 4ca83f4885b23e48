// nr_backward.cu -- fused backward of the rasterize path.
//
// Persistent over the forward's non-empty 16x16 tiles; one thread per internal pixel, a warp owns two
// 16-pixel row segments of the tile (so the pixels of one face form runs in lane order):
//   1. upstream gradient through the 2x2 anti-aliasing mean, flip and permute
//      (autograd of rasterize.py:315-328), read straight from grad_images [B,C,S,S];
//   2. the Differentiation stencil (differentiation.py:13-36, utils.py:75-101) on the
//      internal-resolution image -> d loss / d (x, y) of the pixel;
//   3. coordinate_map backward (rasterize.py:91-97): w_k * grad_xy onto the three vertices of
//      the pixel's face, straight into grad_vertices (the reference goes through a
//      [B,nf,3,3] intermediate and two index_put scatters: rasterize.py:232, utils.py:104-114);
//   4. sample_textures backward (rasterize.py:100-153): bilinear taps into grad_textures, and the
//      perspective-correct uv path into face z and vertices_textures;
//   5. depth-map backward (rasterize.py:80-88) into face z.
// The weight map is a constant for autograd in the reference (it comes out of a CUDA kernel with
// no autograd edge, rasterize.py:75) and is recomputed here from the face instead of being stored.
#include <cudaTypedefs.h>
#include <cstdlib>
#include "nr_kernels.h"

namespace nr {

// d loss / d (x, y) at one pixel. I(c, dy, dx) / G(c, dy, dx) load the image / upstream gradient
// at internal pixel (yi + dy, xi + dx); they are only called for in-range neighbours.
template <class LoadI, class LoadG>
__device__ __forceinline__ void diff_stencil(int yi, int xi, int R, int C, float inv_step, LoadI I,
                                             LoadG G, float &gx, float &gy) {
    const bool ym = yi > 0, yp = yi + 1 < R, xm = xi > 0, xp = xi + 1 < R;
    // r[i] = -sum_c (I[i]-I[i+1]) g[i+1] / step ; l[i] = -sum_c (I[i+1]-I[i]) g[i] / step
    float ry_i = 0.f, ry_m = 0.f, ly_m = 0.f, ly_i = 0.f;
    float rx_i = 0.f, rx_m = 0.f, lx_m = 0.f, lx_i = 0.f;
    for (int c = 0; c < C; ++c) {
        const float ic = I(c, 0, 0), gc = G(c, 0, 0);
        if (yp) {
            const float in = I(c, 1, 0), gn = G(c, 1, 0);
            ry_i = __fadd_rn(ry_i, __fmul_rn(__fsub_rn(ic, in), gn));
            ly_i = __fadd_rn(ly_i, __fmul_rn(__fsub_rn(in, ic), gc));
        }
        if (ym) {
            const float ip = I(c, -1, 0), gp = G(c, -1, 0);
            ry_m = __fadd_rn(ry_m, __fmul_rn(__fsub_rn(ip, ic), gc));
            ly_m = __fadd_rn(ly_m, __fmul_rn(__fsub_rn(ic, ip), gp));
        }
        if (xp) {
            const float in = I(c, 0, 1), gn = G(c, 0, 1);
            rx_i = __fadd_rn(rx_i, __fmul_rn(__fsub_rn(ic, in), gn));
            lx_i = __fadd_rn(lx_i, __fmul_rn(__fsub_rn(in, ic), gc));
        }
        if (xm) {
            const float ip = I(c, 0, -1), gp = G(c, 0, -1);
            rx_m = __fadd_rn(rx_m, __fmul_rn(__fsub_rn(ip, ic), gc));
            lx_m = __fadd_rn(lx_m, __fmul_rn(__fsub_rn(ic, ip), gp));
        }
    }
    // torch divides by the python scalar `step` as a multiplication by 1/step on CUDA
    const float gyr = __fadd_rn(__fmul_rn(-ry_i, inv_step), __fmul_rn(-ry_m, inv_step));
    const float gyl = __fadd_rn(__fmul_rn(-ly_m, inv_step), __fmul_rn(-ly_i, inv_step));
    const float gxr = __fadd_rn(__fmul_rn(-rx_i, inv_step), __fmul_rn(-rx_m, inv_step));
    const float gxl = __fadd_rn(__fmul_rn(-lx_m, inv_step), __fmul_rn(-lx_i, inv_step));
    gy = nr_maximum(gyr, gyl);
    gx = nr_maximum(gxr, gxl);
}

__device__ __forceinline__ int first_argmin3(const float a[3]) {
    int k = 0;
    if (a[1] < a[k]) k = 1;
    if (a[2] < a[k]) k = 2;
    return k;
}
__device__ __forceinline__ int first_argmax3(const float a[3]) {
    int k = 0;
    if (a[1] > a[k]) k = 1;
    if (a[2] > a[k]) k = 2;
    return k;
}

// backward of min(max(x0, lo), hi): gradient shares for x0, lo, hi (ties split evenly, like
// torch.max / torch.min on two tensors)
__device__ __forceinline__ void clamp_shares(float x0, float lo, float hi, float &sx, float &slo,
                                             float &shi) {
    const float x1 = fmaxf(x0, lo);
    float s1 = (x1 < hi) ? 1.f : ((x1 > hi) ? 0.f : 0.5f);
    shi = 1.f - s1;
    const float sa = (x0 > lo) ? 1.f : ((x0 < lo) ? 0.f : 0.5f);
    sx = s1 * sa;
    slo = s1 * (1.f - sa);
}

// Backward of sample_texture(): returns the four tap indices (-1 when the tap reads as zero),
// the tap weights, and the gradients w.r.t. face depths and corner uv's.
template <bool NEED_UV>
__device__ __forceinline__ void sample_texture_backward(const float *__restrict__ tex_b, int H, int W,
                                                        float eps, const float q[3], const float z[3],
                                                        const float u[3], const float v[3], const float *aux,
                                                        const float g_lit[3], const float cw[3], float g[3],
                                                        float rgb_tex[3], int tap[4], float tw[4],
                                                        int &cell, float gz[3], float gu[3], float gv[3]) {
    // exact divisions like the forward: texel coordinates reach ~1e3, where the fast division's 2 ulp
    // would move the bilinear weights by more than the 1e-5 gradient tolerance.  With the forward's aux map
    // the three quotients are read back instead (aux = depth, nx, ny of this pixel).
    const TexCoord tc = aux ? texel_coord_stored(aux[0], aux[1], aux[2], z, u, v, eps) : texel_coord<true>(q, z, u, v, eps);
    const float depth = tc.depth, nx = tc.nx, ny = tc.ny, x0 = tc.x0, y0 = tc.y0, xf = tc.xf, yf = tc.yf;
    const float *zz = tc.zz;
    const float ulo = fminf(u[0], fminf(u[1], u[2])), uhi = __fsub_rn(fmaxf(u[0], fmaxf(u[1], u[2])), eps);
    const float vlo = fminf(v[0], fminf(v[1], v[2])), vhi = __fsub_rn(fmaxf(v[0], fmaxf(v[1], v[2])), eps);
    const float xff = floorf(xf), yff = floorf(yf), xcf = xff + 1.f, ycf = yff + 1.f;
    const int xfi = (int)xff, yfi = (int)yff, xci = (int)xcf, yci = (int)ycf;
    const float ax = xcf - xf, bx = xf - xff, ay = ycf - yf, by = yf - yff;
    tw[0] = ay * ax; tw[1] = ay * bx; tw[2] = by * ax; tw[3] = by * bx;
    const int T = H * W;
    tap[0] = yfi * W + xfi; tap[1] = yfi * W + xci; tap[2] = yci * W + xfi; tap[3] = yci * W + xci;
    cell = (yfi << 16) ^ (xfi & 0xffff);   // identifies the bilinear cell: equal cell => equal four taps
    // g = upstream gradient of the UNLIT sample (lit = unlit * cw, rasterize.py:283); rgb_tex = unlit sample
    float d[4];
    g[0] = g_lit[0] * cw[0]; g[1] = g_lit[1] * cw[1]; g[2] = g_lit[2] * cw[2];
    rgb_tex[0] = rgb_tex[1] = rgb_tex[2] = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        if ((unsigned)tap[t] >= (unsigned)T) tap[t] = -1;
        d[t] = 0.f;
        if (tap[t] >= 0) {
            const float *pt = tex_b + tap[t];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float tv = __ldg(pt + c * T);
                d[t] += g[c] * tv;
                rgb_tex[c] += tw[t] * tv;
            }
        }
    }
    const float gxf = ay * (d[1] - d[0]) + by * (d[3] - d[2]);
    const float gyf = ax * (d[2] - d[0]) + bx * (d[3] - d[1]);
    float sx, sxlo = 0.f, sxhi = 0.f, sy, sylo = 0.f, syhi = 0.f;
    clamp_shares(x0, ulo, uhi, sx, sxlo, sxhi);
    clamp_shares(y0, vlo, vhi, sy, sylo, syhi);
    const float gx0 = gxf * sx, gy0 = gyf * sy;
    const float gnx = gx0 * depth, gny = gy0 * depth;
    const float gdepth = gx0 * nx + gy0 * ny;
    const float gD = -gdepth * depth * depth;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float iz = 1.f / zz[k];
        if (NEED_UV) {
            gu[k] = gnx * q[k] * iz;
            gv[k] = gny * q[k] * iz;
        }
        gz[k] = -(gnx * q[k] * u[k] + gny * q[k] * v[k] + gD * q[k]) * iz * iz;
    }
    if (NEED_UV) {
        // clamp bounds depend on the corner uv's themselves (min / max over the corners)
        gu[first_argmin3(u)] += gxf * sxlo;
        gu[first_argmax3(u)] += gxf * sxhi;
        gv[first_argmin3(v)] += gyf * sylo;
        gv[first_argmax3(v)] += gyf * syhi;
    }
}

// Warp-level segmented sum over runs of equal `key` in lane order (a warp is one image row
// segment, so the pixels of one face / one texel cell form runs).  Afterwards the LAST lane of
// every run holds the run total in v[]; returns true on those lanes.  Fixed summation order.
// Lanes with valid == false never join a run.
template <int N>
__device__ __forceinline__ bool run_reduce(int key, bool valid, float (&v)[N], int lane) {
    const int prev = __shfl_up_sync(0xffffffffu, key, 1);
    const bool prev_valid = __shfl_up_sync(0xffffffffu, (int)valid, 1) != 0;
    // an invalid lane is a run of its own and separates the runs around it
    // runs never cross lane 16 (a warp holds two 16-pixel rows), so four doubling steps suffice
    const bool head = ((lane & 15) == 0) || !valid || !prev_valid || (key != prev);
    const unsigned heads = __ballot_sync(0xffffffffu, head);
    if (heads != 0xffffffffu) {
        const int seg_start = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
#pragma unroll
        for (int d = 1; d < 16; d <<= 1) {
            const bool take = (lane - d >= seg_start);
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const float t = __shfl_up_sync(0xffffffffu, v[i], d);
                if (take) v[i] += t;
            }
        }
    }
    return (lane == 31) || ((heads >> (lane + 1)) & 1u);
}

// C = channel count at compile time (0: read it from the arguments).
// Persistent over the forward's list of non-empty 16x16 tiles (grid-stride); a warp owns two
// 16-pixel row segments of the tile, so the pixels of one face form runs in lane order.
// Accumulate one contribution.  Float atomics (default) commute only up to rounding, so the result
// depends on arrival order; in deterministic mode the value is rounded ONCE to 64-bit fixed point
// (value * 2^k) and added with integer atomics, which are exactly associative: the sum is bit-identical
// from run to run whatever the order.  The warp-level run sums in front of it have a fixed order.
template <bool DET, class Index>
__device__ __forceinline__ void accumulate(float *dst_f, long long *dst_i, Index idx, float v, float scale) {
    if (DET) {
        atomicAdd(reinterpret_cast<unsigned long long *>(dst_i + idx),
                  (unsigned long long)__double2ll_rn((double)v * (double)scale));
    } else {
        atomicAdd(dst_f + idx, v);
    }
}

// Gradient of the light data [L, B, 8] from one warp of one view b (autograd of rasterize.py:256-283 with respect
// to color / direction / alpha).  n = interpolated normal (not renormalised), w = d loss / d colour weight of the
// lane's pixel; lanes with on == false contribute nothing.  Per light (warp-uniform loop):
//   ambient      d color = w
//   directional  d color = w a,  d direction = -(w . color) gate n          (a, gate as in light_weights)
//   specular     d color = w a^alpha,  d alpha = (w . color) a^alpha ln a for a > 0, else 0 (torch's pow backward)
// The parameters of a light are summed over the warp by an xor butterfly (fixed order), then lane i adds parameter i:
// at most 7 accumulations per (warp, light), never one per pixel.
template <bool DET>
__device__ __forceinline__ void light_param_grads(const BackwardArgs &a, int b, int lane, bool on, const float n[3],
                                                  const float w[3]) {
    const LightArgs &L = a.lights;
    for (int l = 0; l < L.num; ++l) {
        const int type = __ldg(L.types + l);
        const int kind = type & 3;
        const size_t o = ((size_t)l * a.B + b) * 8;
        const float *d = L.data + o;
        float p[7] = {w[0], w[1], w[2], 0.f, 0.f, 0.f, 0.f};    // ambient: d color = w
        if (kind != 0) {
            const float cr = __ldg(d), cg = __ldg(d + 1), cb = __ldg(d + 2);
            float dir[3] = {0.f, 0.f, 1.f};
            if (kind == 1) { dir[0] = __ldg(d + 3); dir[1] = __ldg(d + 4); dir[2] = __ldg(d + 5); }
            const float raw = __fadd_rn(__fadd_rn(__fmul_rn(-dir[0], n[0]), __fmul_rn(-dir[1], n[1])), __fmul_rn(-dir[2], n[2]));
            const bool backside = (type & 4) != 0;
            const float av = backside ? fabsf(raw) : fmaxf(raw, 0.f);
            const float gate = backside ? (raw > 0.f ? 1.f : (raw < 0.f ? -1.f : 0.f)) : (raw > 0.f ? 1.f : 0.f);
            const float s = w[0] * cr + w[1] * cg + w[2] * cb;
            float inten = av;
            if (kind == 2) {
                inten = powf(av, __ldg(d + 6));
                p[6] = av > 0.f ? s * inten * logf(av) : 0.f;
            } else {
                p[3] = -s * gate * n[0]; p[4] = -s * gate * n[1]; p[5] = -s * gate * n[2];
            }
            p[0] = w[0] * inten; p[1] = w[1] * inten; p[2] = w[2] * inten;
        }
        if (!on) {
#pragma unroll
            for (int i = 0; i < 7; ++i) p[i] = 0.f;
        }
        // parameters this kind has: colour always, direction for directional, alpha for specular
        const bool has_dir = kind == 1, has_alpha = kind == 2;
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            if ((i >= 3 && i < 6 && !has_dir) || (i == 6 && !has_alpha)) continue;
#pragma unroll
            for (int m = 16; m > 0; m >>= 1) p[i] += __shfl_xor_sync(0xffffffffu, p[i], m);
        }
        float v = p[0];
#pragma unroll
        for (int i = 1; i < 7; ++i)
            if (lane == i) v = p[i];
        const bool mine = lane < 3 || (lane < 6 && has_dir) || (lane == 6 && has_alpha);
        if (mine && v != 0.f) accumulate<DET>(a.grad_light, a.det_light, o + lane, v, a.det_scale);
    }
}

// ---- staged front: a tile's face indices, stencil image and upstream gradient are copied into shared memory by
// TMA one work item ahead, so the 41 tile-shaped loads of a foreground pixel wait on no DRAM latency and hold no
// registers in flight.  Boxes (x = column, y = row, z = view * C + channel), in flipped image coordinates:
//   face_index_map  16 x 16 at (16 tx, 16 ty, b)                                   (not flipped)
//   image           24 x 18 x C at (v0 - 4, u0 - 1, b C)       u0 = R - 16 (ty + 1), v0 = R - 16 (tx + 1)
//   grad_images     24 x 18 x C like the image, or under anti-aliasing 16 x 10 x C at ((v0 >> 1) - 4, (u0 >> 1) - 1)
// i.e. the tile plus its one-pixel stencil halo; the x origin is moved 4 columns left (not 1) to stay 16-byte
// aligned.  TMA fills what lies outside the image with zeros; the stencil never reads it (a neighbour outside the
// image is clamped to the centre).  Two stages per CTA; "full" completes with the TMA bytes, "empty" with one
// arrival per warp, so warps that leave a work item early never wait for each other at a CTA barrier.
constexpr int ST_FIM_BYTES = TILE * TILE * 4;
constexpr int ST_W = 24, ST_H = 18, ST_W_AA = 16, ST_H_AA = 10;
__host__ __device__ inline int st_round(int bytes) { return (bytes + 127) & ~127; }
__host__ __device__ inline int st_img_bytes(int C) { return ST_W * ST_H * C * 4; }
__host__ __device__ inline int st_grad_bytes(int C, bool aa) { return (aa ? ST_W_AA * ST_H_AA : ST_W * ST_H) * C * 4; }
__host__ __device__ inline int st_stage_bytes(int C, bool aa) {
    return ST_FIM_BYTES + st_round(st_img_bytes(C)) + st_round(st_grad_bytes(C, aa));
}
__host__ __device__ inline int st_smem_bytes(int C, bool aa) { return 2 * st_stage_bytes(C, aa) + 4 * 8; }

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n"
        "WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra WAIT;\n}" ::"r"(smem_addr(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *map, int x, int y, int z, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(smem_addr(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(z), "r"(smem_addr(bar))
        : "memory");
}
// one thread: the three boxes of tile (b, tx, ty) into stage `st`, completing `full`
__device__ __forceinline__ void stage_issue(const BackwardArgs &a, unsigned char *st, uint64_t *full, int b, int tx,
                                            int ty, int C, bool aa) {
    const int ib = st_img_bytes(C), gb = st_grad_bytes(C, aa), sh = aa ? 1 : 0;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(full)),
                 "r"(ST_FIM_BYTES + ib + gb) : "memory");
    const int u0 = a.R - TILE * (ty + 1), v0 = a.R - TILE * (tx + 1);
    tma_load_3d(st, &a.map_fim, tx * TILE, ty * TILE, b, full);
    tma_load_3d(st + ST_FIM_BYTES, &a.map_img, v0 - 4, u0 - 1, b * C, full);
    tma_load_3d(st + ST_FIM_BYTES + st_round(ib), &a.map_grad, (v0 >> sh) - 4, (u0 >> sh) - 1, b * C, full);
}
template <bool SMEM>
__device__ __forceinline__ float ld_stencil(const float *p) {
    if (SMEM) return *p;
    return __ldg(p);
}

// AUX: the forward left the normalised weights (and, with colour, the texel coordinate) of every foreground pixel
// in the aux map: nothing of that is re-derived here (9 scattered vertex loads and 12 IEEE divisions less per pixel).
// LGRAD: also sum the gradient of the light data (lit variants, CT = 0, with a.grad_light); a variant of its own, so
// that calls with constant lights run exactly the code they ran before light gradients existed.
// STAGED: the face indices and the stencil operands come from shared memory (staged front above); otherwise from
// global memory (any R, any alignment; NR_FORCE_UNSTAGED_BACKWARD=1).  Both compute bit-identical results.
template <int CT, bool NEED_UV, bool DET, bool AUX, bool LGRAD = false, bool STAGED = false>
__global__ void __launch_bounds__(TILE_THREADS, 4)
k_backward(const __grid_constant__ BackwardArgs a) {
    extern __shared__ __align__(128) unsigned char stage_smem[];
    pdl_wait();         // the forward's maps, tile list and zero-filled accumulators (nr_kernels.h)
    const int lane = threadIdx.x & 31, wrow = threadIdx.x >> 5;
    const int R = a.R, S = a.S, C = CT ? CT : a.C;
    const bool aa = (a.flags & FLAG_AA) != 0;
    const int nt = a.ntx * a.ntx;
    TileList tl;
    if (a.tile_list) tl = open_tile_list(a.tile_list, a.B * nt);
    const int count = a.tile_list ? tl.total : a.B * nt;
    auto tile_of = [&](int work, int &b, int &tx, int &ty) {
        if (a.tile_list) {
            const int4 e = tile_entry(tl, work);
            b = e.x; tx = e.y & 0xffff; ty = e.y >> 16;
        } else {
            b = work / nt;
            const int tile = work - b * nt;
            ty = tile / a.ntx; tx = tile - ty * a.ntx;
        }
    };
    const int stage_bytes = STAGED ? st_stage_bytes(C, aa) : 0;
    uint64_t *full = reinterpret_cast<uint64_t *>(stage_smem + 2 * stage_bytes), *empty = full + 2;
    if (STAGED) {
        if (threadIdx.x == 0) {
            mbar_init(full, 1); mbar_init(full + 1, 1);
            mbar_init(empty, TILE_THREADS / 32); mbar_init(empty + 1, TILE_THREADS / 32);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            if ((int)blockIdx.x < count) {
                int b, tx, ty;
                tile_of(blockIdx.x, b, tx, ty);
                stage_issue(a, stage_smem, full, b, tx, ty, C, aa);
            }
        }
        __syncthreads();    // once, for the barrier initialisation
    }
    for (int work = blockIdx.x, it = 0; work < count; work += gridDim.x, ++it) {
    int b, tx, ty;
    tile_of(work, b, tx, ty);
    // item `it` is in stage s, its (it >> 1)-th use
    const int s = it & 1;
    const unsigned char *st = stage_smem + s * stage_bytes;
    if (STAGED) {
        if (threadIdx.x == 0 && work + (int)gridDim.x < count) {
            // the next item goes into the other stage once every warp is done with item it - 1 there
            if (it > 0) mbar_wait(empty + (s ^ 1), ((it - 1) >> 1) & 1);
            int nb, ntx_, nty;
            tile_of(work + gridDim.x, nb, ntx_, nty);
            stage_issue(a, stage_smem + (s ^ 1) * stage_bytes, full + (s ^ 1), nb, ntx_, nty, C, aa);
        }
        mbar_wait(full + s, (it >> 1) & 1);
    }
    const int lx = lane & 15, ly = wrow * 2 + (lane >> 4);
    const int xi = tx * TILE + lx, yi = ty * TILE + ly;
    const bool valid = (xi < R) && (yi < R);
    const int f = !valid ? -1 : (STAGED ? reinterpret_cast<const int *>(st)[ly * TILE + lx]
                                        : __ldg(a.fim + ((size_t)b * R + yi) * R + xi));
    const bool fg = f >= 0;
    // gradients only reach the mesh through foreground pixels (to_map links nothing else,
    // utils.py:104-114): a warp without any is done with this tile
    if (__ballot_sync(0xffffffffu, fg) == 0u) {
        if (STAGED && lane == 0) mbar_arrive(empty + s);
        continue;
    }

    const int u_ = R - 1 - yi, v_ = R - 1 - xi;
    float gx = 0.f, gy = 0.f;
    float gcen[5] = {0.f, 0.f, 0.f, 0.f, 0.f};   // upstream gradient at this pixel, per channel
    if (fg) {
        // neighbour coordinates, clamped so every load is in range; out-of-range pairs are masked
        const bool has_yp = yi + 1 < R, has_ym = yi > 0, has_xp = xi + 1 < R, has_xm = xi > 0;
        const int u_yp = has_yp ? u_ - 1 : u_, u_ym = has_ym ? u_ + 1 : u_;
        const int v_xp = has_xp ? v_ - 1 : v_, v_xm = has_xm ? v_ + 1 : v_;
        const float gs = aa ? 0.25f : 1.f;   // 2x2 mean backward (rasterize.py:323-328), exact
        const int sh = aa ? 1 : 0;
        // one pointer per array (this pixel, channel 0); neighbours and channels are 32-bit element offsets from it
        // (R <= 32768, so a plane has < 2^31 elements).  Staged: the same offsets within the boxes.
        const float *pI, *pG;
        int rowI, rowG, planeI, planeG;
        if (STAGED) {
            const int u0 = R - TILE * (ty + 1), v0 = R - TILE * (tx + 1);
            const int gw = aa ? ST_W_AA : ST_W, gh = aa ? ST_H_AA : ST_H;
            const float *sI = reinterpret_cast<const float *>(st + ST_FIM_BYTES);
            const float *sG = reinterpret_cast<const float *>(st + ST_FIM_BYTES + st_round(st_img_bytes(C)));
            pI = sI + (u_ - u0 + 1) * ST_W + (v_ - v0 + 4);
            pG = sG + ((u_ >> sh) - (u0 >> sh) + 1) * gw + ((v_ >> sh) - (v0 >> sh) + 4);
            rowI = ST_W; rowG = gw; planeI = ST_W * ST_H; planeG = gw * gh;
        } else {
            pI = a.internal + (size_t)b * C * R * R + (size_t)u_ * R + v_;
            pG = a.grad_images + (size_t)b * C * S * S + (size_t)(u_ >> sh) * S + (v_ >> sh);
            rowI = R; rowG = S; planeI = R * R; planeG = S * S;
        }
        const int dI_yp = (u_yp - u_) * rowI, dI_ym = (u_ym - u_) * rowI, dI_xp = v_xp - v_, dI_xm = v_xm - v_;
        const int dG_yp = ((u_yp >> sh) - (u_ >> sh)) * rowG, dG_ym = ((u_ym >> sh) - (u_ >> sh)) * rowG;
        const int dG_xp = (v_xp >> sh) - (v_ >> sh), dG_xm = (v_xm >> sh) - (v_ >> sh);
        float ry_i = 0.f, ry_m = 0.f, ly_m = 0.f, ly_i = 0.f, rx_i = 0.f, rx_m = 0.f, lx_m = 0.f, lx_i = 0.f;
#pragma unroll
        for (int c = 0; c < (CT ? CT : 5); ++c) {
            if (c < C) {
                const float *Ic = pI + c * planeI, *Gc = pG + c * planeG;
                const float ic = ld_stencil<STAGED>(Ic), iyp = ld_stencil<STAGED>(Ic + dI_yp), iym = ld_stencil<STAGED>(Ic + dI_ym);
                const float ixp = ld_stencil<STAGED>(Ic + dI_xp), ixm = ld_stencil<STAGED>(Ic + dI_xm);
                const float gc = __fmul_rn(ld_stencil<STAGED>(Gc), gs), gyp = __fmul_rn(ld_stencil<STAGED>(Gc + dG_yp), gs);
                const float gym = __fmul_rn(ld_stencil<STAGED>(Gc + dG_ym), gs), gxp = __fmul_rn(ld_stencil<STAGED>(Gc + dG_xp), gs);
                const float gxm = __fmul_rn(ld_stencil<STAGED>(Gc + dG_xm), gs);
                gcen[c] = gc;
                // differentiation.py:19-29; a clamped (out-of-range) neighbour equals the centre, so its
                // difference is exactly zero and the term vanishes like the zero padding does
                ry_i = __fadd_rn(ry_i, __fmul_rn(__fsub_rn(ic, iyp), gyp));
                ly_i = __fadd_rn(ly_i, __fmul_rn(__fsub_rn(iyp, ic), gc));
                ry_m = __fadd_rn(ry_m, __fmul_rn(__fsub_rn(iym, ic), gc));
                ly_m = __fadd_rn(ly_m, __fmul_rn(__fsub_rn(ic, iym), gym));
                rx_i = __fadd_rn(rx_i, __fmul_rn(__fsub_rn(ic, ixp), gxp));
                lx_i = __fadd_rn(lx_i, __fmul_rn(__fsub_rn(ixp, ic), gc));
                rx_m = __fadd_rn(rx_m, __fmul_rn(__fsub_rn(ixm, ic), gc));
                lx_m = __fadd_rn(lx_m, __fmul_rn(__fsub_rn(ic, ixm), gxm));
            }
        }
        const float inv_step = __frcp_rn((float)(2. / R));
        const float gyr = __fadd_rn(__fmul_rn(-ry_i, inv_step), __fmul_rn(-ry_m, inv_step));
        const float gyl = __fadd_rn(__fmul_rn(-ly_m, inv_step), __fmul_rn(-ly_i, inv_step));
        const float gxr = __fadd_rn(__fmul_rn(-rx_i, inv_step), __fmul_rn(-rx_m, inv_step));
        const float gxl = __fadd_rn(__fmul_rn(-lx_m, inv_step), __fmul_rn(-lx_i, inv_step));
        gy = nr_maximum(gyr, gyl);
        gx = nr_maximum(gxr, gxl);
    }
    if (STAGED) {       // the rest of the work item needs nothing from the stage
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + s);
    }

    // ---- per-pixel contributions
    int vid[3] = {0, 0, 0};
    float vg[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // (x, y, z) gradient of the 3 corners
    float tg[12] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // 4 taps x rgb
    int tap[4] = {-1, -1, -1, -1};
    int cell = 0;
    bool has_tex = false;
    // light-parameter gradients: the interpolated normal and d loss / d colour weight of a lit pixel, kept
    // outside the divergent per-pixel code for the warp reduction at the end of the work item
    bool lg_on = false;
    float lg_n[3] = {0.f, 0.f, 0.f}, lg_w[3] = {0.f, 0.f, 0.f};
    // CT = 1 is a lone silhouette or depth channel, CT >= 3 always holds the three colour channels
    const bool rgb = (CT == 1) ? false : ((CT >= 3) ? true : (a.flags & FLAG_RGB) != 0);
    constexpr bool LIT = (CT == 0);      // lights only in the generic variants (keeps the common ones small)
    const bool has_z = rgb || (a.flags & FLAG_DEPTH) != 0;
    if (fg) {
        if (a.faces) {
            vid[0] = __ldg(a.faces + 3 * (size_t)f);
            vid[1] = __ldg(a.faces + 3 * (size_t)f + 1);
            vid[2] = __ldg(a.faces + 3 * (size_t)f + 2);
        } else {
            vid[0] = 3 * f; vid[1] = 3 * f + 1; vid[2] = 3 * f + 2;
        }
        const float *vb = a.verts + (size_t)b * a.nv * 3;
        float Z[3] = {1.f, 1.f, 1.f}, q[3], tcs[3] = {0.f, 0.f, 0.f};
        if (AUX) {
            const float *ap = a.aux + (((size_t)b * R + yi) * R + xi) * (rgb ? 6 : 3);
            if (rgb) {
                const float2 a0 = __ldg(reinterpret_cast<const float2 *>(ap)), a1 = __ldg(reinterpret_cast<const float2 *>(ap) + 1),
                             a2 = __ldg(reinterpret_cast<const float2 *>(ap) + 2);
                q[0] = a0.x; q[1] = a0.y; q[2] = a1.x;
                tcs[0] = a1.y; tcs[1] = a2.x; tcs[2] = a2.y;
            } else {
                q[0] = __ldg(ap); q[1] = __ldg(ap + 1); q[2] = __ldg(ap + 2);
            }
            if (has_z) {
#pragma unroll
                for (int k = 0; k < 3; ++k) Z[k] = __ldg(vb + 3 * (size_t)vid[k] + 2);
            }
        } else {
            float X[3], Y[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                X[k] = __ldg(vb + 3 * (size_t)vid[k]);
                Y[k] = __ldg(vb + 3 * (size_t)vid[k] + 1);
                Z[k] = __ldg(vb + 3 * (size_t)vid[k] + 2);
            }
            const float xp = pix_center(xi, R), yp = pix_center(yi, R);
            raw_weights(xp, yp, X[0], Y[0], X[1], Y[1], X[2], Y[2], q[0], q[1], q[2]);
            normalize_weights<true>(q[0], q[1], q[2]);   // exact: 2 ulp on q move texel coordinates of ~1e3 by 1e-4
        }
        float gz[3] = {0.f, 0.f, 0.f};
        int c0 = 0;
        if (rgb) {
            const float g_lit[3] = {gcen[0], gcen[1], gcen[2]};
            if (g_lit[0] != 0.f || g_lit[1] != 0.f || g_lit[2] != 0.f) {
                const int32_t *fti = a.ft + 3 * (size_t)f;
                const float *vtb = a.vt + (size_t)b * a.nvt * 2;
                int tvid[3];
                float u[3], v[3];
                bool tex_ok = true;      // an out-of-range texture-vertex index contributes nothing (the forward drew black)
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    tvid[k] = __ldg(fti + k);
                    const bool ok = (unsigned)tvid[k] < (unsigned)a.nvt;
                    tex_ok &= ok;
                    if (!ok) tvid[k] = 0;
                    const float2 uv = __ldg(reinterpret_cast<const float2 *>(vtb) + tvid[k]);
                    u[k] = uv.x;
                    v[k] = uv.y;
                }
                if (tex_ok) {
                float gu[3] = {0.f, 0.f, 0.f}, gv[3] = {0.f, 0.f, 0.f}, tw[4], g[3], rgb_tex[3];
                float cw[3] = {1.f, 1.f, 1.f}, nrm[3] = {0.f, 0.f, 0.f};
                const bool lit = LIT && a.lights.num > 0;
                if (lit) {
                    const float *vnb = a.lights.vnormals + (size_t)b * a.nv * 3;
#pragma unroll
                    for (int k = 0; k < 3; ++k)
#pragma unroll
                        for (int c = 0; c < 3; ++c)
                            nrm[c] = __fadd_rn(nrm[c], __fmul_rn(q[k], __ldg(vnb + 3 * (size_t)vid[k] + c)));
                    light_weights(a.lights, b, a.B, nrm, cw, nullptr, nullptr);
                }
                sample_texture_backward<NEED_UV>(a.tex + (size_t)b * 3 * a.H * a.W, a.H, a.W, a.eps, q, Z, u, v, AUX ? tcs : nullptr,
                                        g_lit, cw, g, rgb_tex, tap, tw, cell, gz, gu, gv);
                if (lit && a.lights.grad_vnormals) {
                    // d loss / d colour weight = upstream * unlit sample; then through the lights to the normal
                    const float gcw[3] = {g_lit[0] * rgb_tex[0], g_lit[1] * rgb_tex[1], g_lit[2] * rgb_tex[2]};
                    float cw2[3], gn[3];
                    light_weights(a.lights, b, a.B, nrm, cw2, gcw, gn);
                    const size_t ovn = (size_t)b * a.nv * 3;
#pragma unroll
                    for (int k = 0; k < 3; ++k)
#pragma unroll
                        for (int c = 0; c < 3; ++c)
                            if (gn[c] != 0.f)
                                accumulate<DET>(a.lights.grad_vnormals, a.det_vn, ovn + 3 * (size_t)vid[k] + c, q[k] * gn[c], a.det_scale);
                }
                if (LGRAD && lit) {
                    lg_on = true;
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        lg_n[c] = nrm[c];
                        lg_w[c] = g_lit[c] * rgb_tex[c];
                    }
                }
                has_tex = true;
#pragma unroll
                for (int t = 0; t < 4; ++t)
#pragma unroll
                    for (int c = 0; c < 3; ++c) tg[t * 3 + c] = tw[t] * g[c];
                if (NEED_UV) {
                    const size_t o = (size_t)b * a.nvt * 2;
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        if (gu[k] != 0.f) accumulate<DET>(a.grad_vt, a.det_vt, o + 2 * (size_t)tvid[k], gu[k], a.det_scale);
                        if (gv[k] != 0.f) accumulate<DET>(a.grad_vt, a.det_vt, o + 2 * (size_t)tvid[k] + 1, gv[k], a.det_scale);
                    }
                }
                }   // tex_ok
            }
            c0 = 3;
        }
        if (a.flags & FLAG_SIL) ++c0;
        if (a.flags & FLAG_DEPTH) {
            const float gd = gcen[c0 < 5 ? c0 : 4];
            if (gd != 0.f) {
                const float s = (q[0] / Z[0] + q[1] / Z[1]) + q[2] / Z[2];
                const float dm = 1.f / s;
                const float t = gd * dm * dm;
#pragma unroll
                for (int k = 0; k < 3; ++k) gz[k] += t * q[k] / (Z[k] * Z[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            vg[3 * k] = q[k] * gx;
            vg[3 * k + 1] = q[k] * gy;
            vg[3 * k + 2] = gz[k];
        }
    }

    // ---- vertices: one atomic per (run of equal face, corner, coordinate)
    {
        bool nz = false;
#pragma unroll
        for (int i = 0; i < 9; ++i) nz |= (vg[i] != 0.f);
        if (__ballot_sync(0xffffffffu, nz) != 0u) {
            const bool tail = run_reduce<9>(f, fg, vg, lane);
            if (tail && fg) {
                const size_t o = (size_t)b * a.nv * 3;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const size_t ok = o + 3 * (size_t)vid[k];
                    float *pf = a.grad_verts + ok;
                    long long *pi = DET ? a.det_verts + ok : nullptr;
                    // one test per corner instead of one per component (every tested reduction costs a branch
                    // with a reconvergence barrier); z only moves where there is colour or depth to explain
                    if ((vg[3 * k] != 0.f) | (vg[3 * k + 1] != 0.f) | (vg[3 * k + 2] != 0.f)) {
                        accumulate<DET>(pf, pi, 0, vg[3 * k], a.det_scale);
                        accumulate<DET>(pf, pi, 1, vg[3 * k + 1], a.det_scale);
                        if (has_z) accumulate<DET>(pf, pi, 2, vg[3 * k + 2], a.det_scale);
                    }
                }
            }
        }
    }
    // ---- textures: one atomic per (run of equal base texel, tap, channel)
    if (rgb && a.grad_tex) {
        const bool has = has_tex;
        if (__ballot_sync(0xffffffffu, has) != 0u) {
            const bool tail = run_reduce<12>(cell, has, tg, lane);
            if (tail && has) {
                const size_t T = (size_t)a.H * a.W, o = (size_t)b * 3 * T;
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    if (tap[t] < 0) continue;
                    float *pf = a.grad_tex + o + tap[t];
                    long long *pi = DET ? a.det_tex + o + tap[t] : nullptr;
#pragma unroll
                    for (int c = 0; c < 3; ++c)
                        accumulate<DET>(pf, pi, c * (int)T, tg[t * 3 + c], a.det_scale);
                }
            }
        }
    }
    // ---- light parameters: summed over the warp's 32 pixels, one accumulation per (warp, light, parameter)
    if (LIT && LGRAD && __ballot_sync(0xffffffffu, lg_on) != 0u)
        light_param_grads<DET>(a, b, lane, lg_on, lg_n, lg_w);
    }   // tiles
}

__global__ void __launch_bounds__(256)
k_fixed_to_float(const long long *__restrict__ src, float *__restrict__ dst, size_t n, float inv_scale) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] += (float)((double)src[i] * (double)inv_scale);
}

// Differentiation.backward on channels-last tensors (the public differentiation() op).
__global__ void __launch_bounds__(256)
k_differentiation_backward(const float *__restrict__ images, const float *__restrict__ grad_out,
                           float *__restrict__ grad_xy, int B, int R, int C) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)B * R * R;
    if (i >= total) return;
    const int xi = (int)(i % R), yi = (int)((i / R) % R);
    const float *Ib = images + (size_t)i * C;
    const float *Gb = grad_out + (size_t)i * C;
    auto LI = [&](int c, int dy, int dx) -> float { return __ldg(Ib + ((long long)dy * R + dx) * C + c); };
    auto LG = [&](int c, int dy, int dx) -> float { return __ldg(Gb + ((long long)dy * R + dx) * C + c); };
    const float inv_step = __frcp_rn((float)(2. / R));
    float gx, gy;
    diff_stencil(yi, xi, R, C, inv_step, LI, LG, gx, gy);
    grad_xy[i * 2] = gx;
    grad_xy[i * 2 + 1] = gy;
}

// cuTensorMapEncodeTiled from the driver through the runtime (no -lcuda); null if the driver has none
static PFN_cuTensorMapEncodeTiled_v12000 tensor_map_encoder() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &p, 12000, cudaEnableDefault, &q) != cudaSuccess) {
            cudaGetLastError();     // not an error of the caller's work: the unstaged path runs instead
            p = nullptr;
        }
        if (q != cudaDriverEntryPointSuccess) p = nullptr;
        return reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
    }();
    return fn;
}

// [planes, rows, cols] tensor of 4-byte elements, row-major, box (bx, by, bz); false where TMA cannot address it
static bool encode_map(CUtensorMap *m, CUtensorMapDataType type, const void *base, long long planes, int rows, int cols,
                       int bx, int by, int bz) {
    const cuuint64_t dim[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)planes};
    const cuuint64_t stride[2] = {(cuuint64_t)cols * 4, (cuuint64_t)cols * rows * 4};
    const cuuint32_t box[3] = {(cuuint32_t)bx, (cuuint32_t)by, (cuuint32_t)bz}, estride[3] = {1, 1, 1};
    return tensor_map_encoder()(m, type, 3, const_cast<void *>(base), dim, stride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Tensor maps of the staged front into s; false when TMA's rules rule it out (a row stride that is not a multiple
// of 16 bytes, a base pointer that is not 16-byte aligned), or when NR_FORCE_UNSTAGED_BACKWARD=1 asks for the
// unstaged path (read at every call, so that a test can run both).
static bool prepare_staging(BackwardArgs &s) {
    const char *force = getenv("NR_FORCE_UNSTAGED_BACKWARD");
    if (force && atoi(force) != 0) return false;
    const bool aa = (s.flags & FLAG_AA) != 0;
    auto aligned = [](const void *p) { return ((uintptr_t)p & 15) == 0; };
    if (s.R % 4 || s.S % 4 || !aligned(s.fim) || !aligned(s.internal) || !aligned(s.grad_images) || !tensor_map_encoder())
        return false;
    return encode_map(&s.map_fim, CU_TENSOR_MAP_DATA_TYPE_INT32, s.fim, s.B, s.R, s.R, TILE, TILE, 1) &&
           encode_map(&s.map_img, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, s.internal, (long long)s.B * s.C, s.R, s.R, ST_W, ST_H, s.C) &&
           encode_map(&s.map_grad, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, s.grad_images, (long long)s.B * s.C, s.S, s.S,
                      aa ? ST_W_AA : ST_W, aa ? ST_H_AA : ST_H, s.C);
}

template <int CT, bool NEED_UV, bool DET, bool AUX, bool LGRAD = false>
static void launch_variant(const BackwardArgs &a, bool staged, int grid, cudaStream_t stream) {
    const long long px = (long long)a.B * a.R * a.R;
    if (staged)
        launch_after(2, px, k_backward<CT, NEED_UV, DET, AUX, LGRAD, true>, dim3(grid), dim3(TILE_THREADS),
                     (size_t)st_smem_bytes(a.C, (a.flags & FLAG_AA) != 0), stream, a);
    else
        launch_after(2, px, k_backward<CT, NEED_UV, DET, AUX, LGRAD, false>, dim3(grid), dim3(TILE_THREADS), 0, stream, a);
}

cudaError_t launch_backward(const BackwardArgs &args, cudaStream_t stream) {
    if (args.B <= 0 || args.R <= 0) return cudaSuccess;
    BackwardArgs a = args;
    // Lit calls with constant lights keep the unstaged path: staged, lit config 2 measured 0.4 % slower per step, while
    // with light gradients it measured 0.3 % faster (profiles/r4_backward_staging_lit.txt).
    const bool const_lights = a.lights.num > 0 && !a.grad_light;
    const bool staged = !const_lights && prepare_staging(a);
    const long long tiles = (long long)a.ntx * a.ntx * a.B;
    // exactly the resident CTAs (4 per SM): a second wave of the static tile stride only adds a tail
    const int grid = (int)(tiles < (long long)a.sm_count * 4 ? tiles : (long long)a.sm_count * 4);
    ProfScope p(PROF_BACKWARD, stream);
    if (a.grad_light && a.lights.num > 0) {
        // light gradients: the lit variants with the light-parameter reduction (a.C does not matter: CT = 0)
        if (a.det_verts) {
            if (a.grad_vt) launch_variant<0, true, true, false, true>(a, staged, grid, stream);
            else launch_variant<0, false, true, false, true>(a, staged, grid, stream);
        } else if (a.grad_vt) {
            if (a.aux) launch_variant<0, true, false, true, true>(a, staged, grid, stream);
            else launch_variant<0, true, false, false, true>(a, staged, grid, stream);
        } else {
            if (a.aux) launch_variant<0, false, false, true, true>(a, staged, grid, stream);
            else launch_variant<0, false, false, false, true>(a, staged, grid, stream);
        }
    } else if (a.det_verts) {
        if (a.grad_vt) launch_variant<0, true, true, false>(a, staged, grid, stream);
        else launch_variant<0, false, true, false>(a, staged, grid, stream);
    } else if (a.grad_vt) {
        if (a.aux) launch_variant<0, true, false, true>(a, staged, grid, stream);
        else launch_variant<0, true, false, false>(a, staged, grid, stream);
    } else if (a.aux) {
        switch (a.lights.num > 0 ? 0 : a.C) {
            case 1: launch_variant<1, false, false, true>(a, staged, grid, stream); break;
            case 3: launch_variant<3, false, false, true>(a, staged, grid, stream); break;
            case 4: launch_variant<4, false, false, true>(a, staged, grid, stream); break;
            default: launch_variant<0, false, false, true>(a, staged, grid, stream); break;
        }
    } else {
        switch (a.lights.num > 0 ? 0 : a.C) {
            case 1: launch_variant<1, false, false, false>(a, staged, grid, stream); break;
            case 3: launch_variant<3, false, false, false>(a, staged, grid, stream); break;
            case 4: launch_variant<4, false, false, false>(a, staged, grid, stream); break;
            default: launch_variant<0, false, false, false>(a, staged, grid, stream); break;
        }
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess || !a.det_verts) return e;
    // fixed point -> float, added onto the caller's (zero-filled) gradient tensors
    const float inv = 1.f / a.det_scale;
    auto conv = [&](const long long *src, float *dst, size_t n) {
        if (src && dst && n) k_fixed_to_float<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(src, dst, n, inv);
    };
    conv(a.det_verts, a.grad_verts, (size_t)a.B * a.nv * 3);
    conv(a.det_tex, a.grad_tex, (size_t)a.B * 3 * a.H * a.W);
    conv(a.det_vt, a.grad_vt, (size_t)a.B * a.nvt * 2);
    conv(a.det_vn, a.lights.grad_vnormals, (size_t)a.B * a.nv * 3);
    conv(a.det_light, a.grad_light, (size_t)a.lights.num * a.B * 8);
    return cudaGetLastError();
}

cudaError_t launch_differentiation_backward(const float *images, const float *grad_output,
                                            float *grad_coordinates, int B, int R, int C,
                                            cudaStream_t stream) {
    const long long total = (long long)B * R * R;
    if (total <= 0) return cudaSuccess;
    ProfScope p(PROF_DIFF_BACKWARD, stream);
    k_differentiation_backward<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(
        images, grad_output, grad_coordinates, B, R, C);
    return cudaGetLastError();
}

}  // namespace nr
