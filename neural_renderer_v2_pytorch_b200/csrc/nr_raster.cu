// nr_raster.cu -- tile rasterizer with fused shading epilogue.
//
// Persistent kernel: one WARP owns an 8x4 pixel block of a non-empty tile (16x16, or 8x8 for dense
// meshes), claimed dynamically from the heavy-first tile list.  It walks the tile's face list
// (ascending face index) 32 entries at a time: one lane per face culls against the block (pixel box,
// then a conservative edge-interval test, ballot), the survivors are staged in the warp's slice of
// shared memory, and only those are evaluated per pixel with the reference's arithmetic:
//   rasterize_cuda_kernel.cu:94-149  (z-buffer, sequential 1e-4 hysteresis)
// The epilogue fuses what the reference does in ~60 torch ops and 9*B host round trips:
//   rasterize_cuda_kernel.cu:246-308 weight map, rasterize.py:100-153 texture sampling,
//   :240-242 silhouettes, :80-88 depth, :295-310 channel merge, :315-316 permute + flip,
//   :321-328 2x2 anti-aliasing mean.
#include "nr_shade.cuh"

namespace nr {

// Conservative test "no pixel of the block [xa, xb] x [ya, yb] (pixel-centre coordinates) can pass
// the reference's inside test for this face" (rasterize_cuda_kernel.cu:107-116).  The reference accepts
// a pixel iff c1*c2 >= 0 and c2*c3 >= 0 in float arithmetic, which also lets every pixel with c2 == 0
// (or an underflowing product) through.  So a block is only rejected when, over the whole block, c2
// is bounded away from zero AND c1 or c3 is bounded away from zero with the opposite sign.  The edge
// functions are affine, so their range over the block is spanned by the four corners; the bounds
// carry a margin 40x above the rounding error of the reference's float evaluation.  NaN never rejects.
__device__ __forceinline__ bool block_outside_face(float x0, float y0, float x1, float y1, float x2,
                                                   float y2, float xa, float xb, float ya, float yb) {
    const float dx10 = x1 - x0, dy10 = y1 - y0, dx21 = x2 - x1, dy21 = y2 - y1, dx02 = x0 - x2, dy02 = y0 - y2;
    float lo1, hi1, lo2, hi2, lo3, hi3;
    {
        const float a = (ya - y0) * dx10, b = (yb - y0) * dx10, c = dy10 * (xa - x0), d = dy10 * (xb - x0);
        lo1 = fminf(a, b) - fmaxf(c, d);
        hi1 = fmaxf(a, b) - fminf(c, d);
        const float m = 1e-5f * (fmaxf(fabsf(a), fabsf(b)) + fmaxf(fabsf(c), fabsf(d))) + 1e-30f;
        lo1 -= m;
        hi1 += m;
    }
    {
        const float a = (ya - y1) * dx21, b = (yb - y1) * dx21, c = dy21 * (xa - x1), d = dy21 * (xb - x1);
        lo2 = fminf(a, b) - fmaxf(c, d);
        hi2 = fmaxf(a, b) - fminf(c, d);
        const float m = 1e-5f * (fmaxf(fabsf(a), fabsf(b)) + fmaxf(fabsf(c), fabsf(d))) + 1e-30f;
        lo2 -= m;
        hi2 += m;
    }
    {
        const float a = (ya - y2) * dx02, b = (yb - y2) * dx02, c = dy02 * (xa - x2), d = dy02 * (xb - x2);
        lo3 = fminf(a, b) - fmaxf(c, d);
        hi3 = fmaxf(a, b) - fminf(c, d);
        const float m = 1e-5f * (fmaxf(fabsf(a), fabsf(b)) + fmaxf(fabsf(c), fabsf(d))) + 1e-30f;
        lo3 -= m;
        hi3 += m;
    }
    const bool c2pos = lo2 > 0.f, c2neg = hi2 < 0.f;
    return (c2pos && (hi1 < 0.f || hi3 < 0.f)) || (c2neg && (lo1 > 0.f || lo3 > 0.f));
}


// Persistent kernel over the non-empty tiles.  The unit of work is one WARP = one 8x8 pixel block
// of a tile, two pixels per lane: lane l owns (l & 7, l >> 3) of the upper 8x4 half and the pixel four rows
// below it in the lower half.  A block is claimed from a per-CTA cursor (see "Scheduling"); the blocks of a
// tile are neighbours in the claim order, so its records are shared through L1 / L2.  Warps never wait for
// each other: a block without candidate faces costs one cull pass.
// Per 32 faces of the tile list: every lane loads one face record, tests its pixel box against the
// block, the survivors are compacted (ballot) into this warp's slice of shared memory with their edge
// deltas and their pixel box as a bit mask over each half, then evaluated per pixel in list order.
// Culling 8x8 blocks instead of 8x4 halves the cull, compaction and claim work per pixel; the edge
// functions are still evaluated only for the faces whose box touches the pixel's half.
// Every pixel of the block is written (background included), see "output initialisation" above.
constexpr int RASTER_WARPS = TILE_THREADS / 32;
constexpr int BLK = 8;          // a warp's block is BLK x BLK pixels, in two 8x4 halves
constexpr int HALF_H = 4;

// NR_LAZY_Z: the z-test of a REGULAR candidate (face_z_regular, weights_one_sign: nothing cancels) is decided
// with fast_zp() whenever the outcome is clear of its error bound, which it is for everything but near-ties:
// the seven IEEE divisions of the reference's depth (~65 instructions) are then never executed.  The running
// minimum may therefore be the cheap depth of the current winner (dexact == false); the first comparison that
// is not clear recomputes it exactly from the winner's weights, so every DECISION equals the reference's.
#ifndef NR_LAZY_Z
#define NR_LAZY_Z 1
#endif
constexpr int REC_Q = NR_LAZY_Z ? 5 : 4;       // float4 per staged face

__device__ __noinline__ float exact_zp_call(float w0, float w1, float w2, float z0, float z1, float z2) {
    return exact_zp(w0, w1, w2, z0, z1, z2);
}

// z-buffer state of one pixel: the running minimum, whether it is the reference's exact value, the winner.
// The winner's raw weights and corner depths are not carried: they are recomputed from its record
// (winner_weights) where they are needed, with the same arithmetic on the same floats.
struct ZPix {
    float depth_min;
    bool dexact;
    int best;
};

// raw weight numerators at (xp, yp) and corner depths of face f (its record, rasterize_cuda_kernel.cu:129-132)
__device__ __forceinline__ void winner_weights(const FaceRec *rec_b, int f, float xp, float yp, float &w0, float &w1,
                                               float &w2, float &z0, float &z1, float &z2) {
    const float4 *rp = reinterpret_cast<const float4 *>(rec_b + f);
    const float4 q0 = __ldg(rp), q1 = __ldg(rp + 1);
    z2 = __ldg(reinterpret_cast<const float *>(rp + 2));
    raw_weights(xp, yp, q0.x, q0.y, q0.w, q1.x, q1.z, q1.w, w0, w1, w2);
    z0 = q0.z;
    z1 = q1.y;
}

// the reference's inside test (rasterize_cuda_kernel.cu:107-116) against a staged face
__device__ __forceinline__ bool edge_inside(float xp, float yp, const float4 &A, const float4 &Bq, const float4 &Cq) {
    const float c1 = __fmaf_rn(__fsub_rn(yp, A.y), Bq.z, -__fmul_rn(Bq.w, __fsub_rn(xp, A.x)));
    const float c2 = __fmaf_rn(__fsub_rn(yp, A.w), Cq.x, -__fmul_rn(Cq.y, __fsub_rn(xp, A.z)));
    const float c3 = __fmaf_rn(__fsub_rn(yp, Bq.y), Cq.z, -__fmul_rn(Cq.w, __fsub_rn(xp, Bq.x)));
    return !((__fmul_rn(c1, c2) < 0.f) | (__fmul_rn(c2, c3) < 0.f));
}

// Variants: RGB (texture sampling), AA (2x2 mean epilogue), FULL (everything optional: lights,
// backgrounds, the weight / depth maps of rasterize_maps, resolutions that are no multiple of 16).
// The plain variants leave that code out, which halves their size: at 75 KB the one-size kernel spent
// as many issue slots waiting for instructions as for memory.  TEX: the texture kind (per-face cubes: FULL only).
template <bool RGB, bool AA, bool FULL, bool FINE, int TEX = TEX_UV>
__global__ void __launch_bounds__(TILE_THREADS, 4)
k_raster(const RasterArgs a) {
    pdl_wait();         // the binning kernel's records, lists and header (nr_kernels.h)
    pdl_trigger();      // the backward may be scheduled as this kernel's CTAs leave
    constexpr int TSZ = FINE ? FINE_TILE : TILE;
    __shared__ float4 s_rec[RASTER_WARPS][32][REC_Q];
    __shared__ uint2 s_bb[RASTER_WARPS][32];

    // If the pair list did not fit the workspace, the lists are unusable: every block then scans ALL
    // faces of its view (the records are complete regardless), which is the reference's own loop with
    // the block cull in front.  Slow but correct, and the host grows the workspace for the next call.
    const bool overflow = a.hdr->overflow != 0;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int R = a.R;
    const TileList tl = open_tile_list(a.tile_list, a.B * a.ntx * a.ntx);
    // A tile is 16x16 pixels = 4 warp blocks of 8x8, or in the FINE variants 8x8 = 1 block.  When even the
    // 8x4 blocks of all tiles fit in one wave of resident warps (e.g. a single view), the kernel is bound by
    // the latency of its slowest block, not by issue: it then runs 8x4 blocks (the lower pixel of a lane
    // idles), 8 per 16x16 tile or 2 per 8x8 tile, and a warp has half the pixels to walk in series.
    const bool tall = (long long)tl.total * (FINE ? 2 : 8) > (long long)a.sm_count * 4 * RASTER_WARPS;
    const int bh = tall ? BLK : HALF_H;                                   // block height
    const int blk_shift = (FINE ? 0 : 2) + (tall ? 0 : 1), items = tl.total << blk_shift;
    const bool has_bg = FULL && RGB && a.lights.backgrounds != nullptr;
    const PixGrid grid(R);
    const unsigned lt_mask = (1u << lane) - 1u;
    float4 (*my_rec)[REC_Q] = s_rec[wid];
    uint2 *my_bb = s_bb[wid];

    // ---- fill items (stores only, nr_shade.cuh), interleaved with the raster items: claim i also performs
    // fill item i (a static share per warp was slower: the warps holding the heavy tiles kept their fills
    // for the end)
    const FillPlan plan = make_fill_plan(a);
    const int fill_items = plan.fill_items;

    // Scheduling: the CTA claims EIGHT consecutive items (the blocks of two 16x16 tiles, of one with 8x4 blocks) with one global
    // atomicAdd and its warps take them one by one from a shared cursor, so the blocks of a tile run on the
    // same SM at about the same time (face records and lists shared through L1) and no warp waits for
    // another except while a batch is being fetched.  One shared word holds both the batch and the number
    // of items taken from it: s_cur = (first item of the batch / 8) << 5 | taken; the warp that draws
    // taken == 8 fetches the next batch, later ones (at most 7: 5 bits are plenty) wait for it.
    constexpr int GRAB = 1, BATCH = 8;
    __shared__ unsigned s_cur;
    const int all_items = max(items, fill_items);
    if (threadIdx.x == 0) s_cur = ((unsigned)atomicAdd(&a.hdr->work_counter, BATCH) >> 3) << 5;
    __syncthreads();
    while (true) {
        int first = 0;
        if (lane == 0) {
            while (true) {
                const unsigned v = atomicAdd(&s_cur, 1u);
                const unsigned taken = v & 31u;
                if (taken < BATCH) {
                    first = (int)((v >> 5) << 3) + (int)taken;
                    break;
                }
                if (taken == BATCH) {
                    const unsigned base = (unsigned)atomicAdd(&a.hdr->work_counter, BATCH);
                    atomicExch(&s_cur, (base >> 3) << 5);
                } else {
                    while ((*reinterpret_cast<volatile unsigned *>(&s_cur) >> 5) == (v >> 5)) { }
                }
            }
        }
        first = __shfl_sync(0xffffffffu, first, 0);
        if (first >= all_items) break;
        if (first < fill_items) do_fill_item<AA, FULL, FINE>(a, plan, first, lane);
    for (int item = first; item < min(first + GRAB, items); ++item) {
        const int4 e0 = tile_entry(tl, item >> blk_shift);
        const int sub = item & ((1 << blk_shift) - 1);
        const int b = e0.x, n = overflow ? a.nf : e0.w;
        const int32_t *list = a.pairs + e0.z;
        const int wx0 = (e0.y & 0xffff) * TSZ + (FINE ? 0 : (sub & 1) * BLK), wx1 = wx0 + BLK - 1;
        const int wy0 = (e0.y >> 16) * TSZ + (FINE ? sub : (sub >> 1)) * bh, wy1 = wy0 + bh - 1;
        // this lane's pixels: (xi, yi) in the upper half, (xi, yi + HALF_H) in the lower one
        const int xi = wx0 + (lane & 7), yi = wy0 + (lane >> 3);
        const float xp = grid.center(xi);
        const float yp_u = grid.center(yi), yp_l = grid.center(yi + HALF_H);
        const FaceRec *rec_b = a.rec + (size_t)b * a.nf;
        // pixel centres of the block's corner pixels, for the conservative edge cull
        const float xa = grid.center(wx0), xb = grid.center(wx1);
        const float ya = grid.center(wy0), yb = grid.center(wy1);

        ZPix z_u = {a.far_plane, true, -1}, z_l = z_u;       // upper and lower pixel

        // software pipeline over the list: while group g is culled and evaluated, the records of
        // group g+1 and the ids of group g+2 are already in flight
        auto load_id = [&](int i) -> int { return i < n ? (overflow ? i : __ldg(list + i)) : -1; };
        int fid_next = load_id(lane);
        int fid_next2 = load_id(32 + lane);
        float4 n0 = make_float4(0.f, 0.f, 0.f, 0.f), n1 = n0, n2 = n0;
        if (fid_next >= 0) {
            const float4 *rp = reinterpret_cast<const float4 *>(rec_b + fid_next);
            n0 = __ldg(rp); n1 = __ldg(rp + 1); n2 = __ldg(rp + 2);
        }
        for (int g = 0; g < n; g += 32) {
            // ---- one face per lane: cull against this warp's block, compact the survivors
            const int fid = fid_next;
            const float4 q0 = n0, q1 = n1, q2 = n2;
            fid_next = fid_next2;
            if (fid_next >= 0) {
                const float4 *rp = reinterpret_cast<const float4 *>(rec_b + fid_next);
                n0 = __ldg(rp); n1 = __ldg(rp + 1); n2 = __ldg(rp + 2);
            }
            fid_next2 = load_id(g + 64 + lane);
            bool hit = false;
            if (fid >= 0) {
                const uint32_t bx = __float_as_uint(q2.y), by = __float_as_uint(q2.z);
                hit = ((int)(bx & 0xffff) <= wx1) && ((int)(bx >> 16) >= wx0) && ((int)(by & 0xffff) <= wy1) &&
                      ((int)(by >> 16) >= wy0);
                if (hit) hit = !block_outside_face(q0.x, q0.y, q0.w, q1.x, q1.z, q1.w, xa, xb, ya, yb);
            }
            const unsigned m = __ballot_sync(0xffffffffu, hit);
            if (m == 0u) continue;
            if (hit) {
                const int slot = __popc(m & lt_mask);      // keeps list order
                const float x0 = q0.x, y0 = q0.y, z0 = q0.z, x1 = q0.w;
                const float y1 = q1.x, z1 = q1.y, x2 = q1.z, y2 = q1.w, z2 = q2.x;
                my_rec[slot][0] = make_float4(x0, y0, x1, y1);
                my_rec[slot][1] = make_float4(x2, y2, __fsub_rn(x1, x0), __fsub_rn(y1, y0));
                my_rec[slot][2] = make_float4(__fsub_rn(x2, x1), __fsub_rn(y2, y1), __fsub_rn(x0, x2), __fsub_rn(y0, y2));
                my_rec[slot][3] = make_float4(z0, z1, z2, __int_as_float(fid));
#if NR_LAZY_Z
                // reciprocal depths and the smallest corner depth of a regular face (NaN marks an irregular one)
                const bool zreg = face_z_regular(z0, z1, z2);
                my_rec[slot][4] = make_float4(fast_rcp(z0), fast_rcp(z1), fast_rcp(z2),
                                              zreg ? fminf(z0, fminf(z1, z2)) : __int_as_float(0x7fc00000));
#endif
                // the face's pixel box (:94-97, exact by construction) as a bit mask over this block's 64
                // pixels (bit = lane in .x for the upper half, in .y for the lower one): the columns / rows it
                // covers, relative to the block origin.  A half's word is zero iff the box misses that half.
                const uint32_t bx = __float_as_uint(q2.y), by = __float_as_uint(q2.z);
                const int c0 = max((int)(bx & 0xffff) - wx0, 0), c1 = min((int)(bx >> 16) - wx0, BLK - 1);
                const int r0 = max((int)(by & 0xffff) - wy0, 0), r1 = min((int)(by >> 16) - wy0, bh - 1);
                const uint32_t cols = ((2u << c1) - 1u) & ~((1u << c0) - 1u);          // 8 bits
                const uint32_t rows = ((2u << r1) - 1u) & ~((1u << r0) - 1u);          // 8 bits, 4 per half
                // row r of a half -> bits 8r .. 8r+7
                my_bb[slot] = make_uint2(cols * (((rows & 15u) * 0x00204081u) & 0x01010101u),
                                         cols * (((rows >> 4) * 0x00204081u) & 0x01010101u));
            }
            __syncwarp();
            const int nh = __popc(m);
            // ---- phase 1: coverage of every surviving face, one bit per face and pixel.  Every survivor's box
            // touches at least one half; the record is read once for both.
            unsigned in_u = 0u, in_l = 0u;
            for (int j = 0; j < nh; ++j) {
                const uint2 bb = my_bb[j];       // the same words in every lane: the branches below do not diverge
                const float4 A = my_rec[j][0], Bq = my_rec[j][1], Cq = my_rec[j][2];
                if (bb.x != 0u && (((bb.x >> lane) & 1u) != 0u) & edge_inside(xp, yp_u, A, Bq, Cq)) in_u |= 1u << j;
                if (bb.y != 0u && (((bb.y >> lane) & 1u) != 0u) & edge_inside(xp, yp_l, A, Bq, Cq)) in_l |= 1u << j;
            }
            // ---- phase 2: every lane walks ITS OWN covering faces in list order (the z-test is
            // sequential per pixel only), so lanes evaluate different faces at the same time and the
            // loop runs max-depth-complexity times instead of once per surviving face; a lane walks its
            // upper pixel's faces, then its lower pixel's
#pragma unroll 1
            for (int h = 0; h < 2; ++h) {
                unsigned in = h ? in_l : in_u;
                const float ypp = h ? yp_l : yp_u;
                ZPix z = h ? z_l : z_u;
                while (in) {
                    const int j = __ffs(in) - 1;
                    in &= in - 1;
                    const float4 D = my_rec[j][3];
#if NR_LAZY_Z
                    const float4 E = my_rec[j][4];
                    // surely depth_min < every corner depth (:124-126 skips the face); false for an irregular face
                    if (z.depth_min * (1.f + FAST_Z_REL) < E.w) continue;
                    const float4 A = my_rec[j][0], Bq = my_rec[j][1];
                    float w0, w1, w2;
                    raw_weights(xp, ypp, A.x, A.y, A.z, A.w, Bq.x, Bq.y, w0, w1, w2);
                    if (E.w == E.w && weights_one_sign(w0, w1, w2)) {
                        const float zf = fast_zp(w0, w1, w2, E.x, E.y, E.z);
                        const float mg = 2.f * FAST_Z_REL * fmaxf(zf, z.depth_min);   // error of zf plus that of depth_min
                        const float t = z.depth_min - a.delta;
                        // (every comparison is false for a NaN: such a candidate takes the exact path)
                        if (zf < a.near_plane - mg || zf > a.far_plane + mg || zf > t + mg) continue;   // :140-148 reject it
                        if (zf > a.near_plane + mg && zf < a.far_plane - mg && zf < t - mg) {           // ... accept it
                            z.depth_min = zf;
                            z.dexact = false;
                            z.best = __float_as_int(D.w);
                            continue;
                        }
                    }
                    // not clear: the reference's own arithmetic, against the exact running minimum (the
                    // winner's record is read again: this only runs for near-ties)
                    if (!z.dexact) {
                        float v0, v1, v2, u0, u1, u2;
                        winner_weights(rec_b, z.best, xp, ypp, v0, v1, v2, u0, u1, u2);
                        z.depth_min = exact_zp_call(v0, v1, v2, u0, u1, u2);
                        z.dexact = true;
                    }
                    if (z.depth_min < D.x && z.depth_min < D.y && z.depth_min < D.z) continue;    // :124-126
                    const float zp = exact_zp_call(w0, w1, w2, D.x, D.y, D.z);                      // :129-139
#else
                    // :124-126
                    if (z.depth_min < D.x && z.depth_min < D.y && z.depth_min < D.z) continue;
                    const float4 A = my_rec[j][0], Bq = my_rec[j][1];
                    // :129-136
                    float w0, w1, w2;
                    raw_weights(xp, ypp, A.x, A.y, A.z, A.w, Bq.x, Bq.y, w0, w1, w2);
                    const float zp = exact_zp(w0, w1, w2, D.x, D.y, D.z);
#endif
                    // :139-142
                    if (zp <= a.near_plane || a.far_plane <= zp) continue;
                    // :145-148
                    if (zp <= __fsub_rn(z.depth_min, a.delta)) {
                        z.depth_min = zp;
                        z.best = __float_as_int(D.w);
                    }
                }
                if (h) z_l = z;
                else z_u = z;
            }
            __syncwarp();
        }
        // ---------------------------------------------- epilogue: every pixel of the block is written, one
        // 8x4 half at a time (shade_block's lane layout, its anti-aliasing quads lie within a half)
#pragma unroll 1
        for (int h = 0; h < (tall ? 2 : 1); ++h) {
            const int yh = yi + h * HALF_H, best = h ? z_l.best : z_u.best;
            float bw0 = 0.f, bw1 = 0.f, bw2 = 0.f, bz0 = 0.f, bz1 = 0.f, bz2 = 0.f;
            if (best >= 0) winner_weights(rec_b, best, xp, h ? yp_l : yp_u, bw0, bw1, bw2, bz0, bz1, bz2);
            shade_block<RGB, AA, FULL, TEX>(a, b, xi, yh, (xi < R) && (yh < R), best, bw0, bw1, bw2, bz0, bz1, bz2, has_bg);
        }
    }   // items of this claim
    }   // claims
}

// compute_weight_map_c compatibility kernel (rasterize_cuda_kernel.cu:246-308): one thread per
// pixel, faces given as the gathered [B, nf, 3, 3] tensor, background pixels untouched.
__global__ void __launch_bounds__(256)
k_weight_map_compat(const float *__restrict__ faces, const int32_t *__restrict__ fim,
                    float *__restrict__ wmap, long long total, int nf, int R) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int fi = fim[i];
    if (fi < 0) return;
    const long long pp = (long long)R * R;
    const int bn = (int)(i / pp), pn = (int)(i % pp);
    const int yi = pn / R, xi = pn % R;
    const float xp = pix_center(xi, R), yp = pix_center(yi, R);
    const float *f = faces + ((size_t)bn * nf + fi) * 9;
    float w0, w1, w2;
    raw_weights(xp, yp, f[0], f[1], f[3], f[4], f[6], f[7], w0, w1, w2);
    normalize_weights(w0, w1, w2);
    wmap[i * 3 + 0] = w0;
    wmap[i * 3 + 1] = w1;
    wmap[i * 3 + 2] = w2;
}

// The optional per-pixel maps (weight_map, depth_map: rasterize_maps / the compat operators, not
// on the hot path) are written for foreground pixels only, so they start as zeros.
cudaError_t launch_background_fill(const RasterArgs &a, cudaStream_t stream) {
    if (a.B <= 0 || a.R <= 0 || (!a.wmap && !a.dmap)) return cudaSuccess;
    ProfScope p(PROF_MEMSET, stream);
    const size_t P = (size_t)a.B * a.R * a.R;
    cudaError_t e = cudaSuccess;
    if (a.wmap) e = cudaMemsetAsync(a.wmap, 0, P * 3 * sizeof(float), stream);
    if (e == cudaSuccess && a.dmap) e = cudaMemsetAsync(a.dmap, 0, P * sizeof(float), stream);
    return e;
}

cudaError_t launch_raster(const RasterArgs &a, cudaStream_t stream) {
    if (a.B <= 0 || a.R <= 0) return cudaSuccess;
    const long long tiles = (long long)a.ntx * a.ntx * a.B;
    const int grid = (int)(tiles < (long long)a.sm_count * 8 ? tiles : (long long)a.sm_count * 8);
    const bool rgb = (a.flags & FLAG_RGB) != 0, aa = (a.flags & FLAG_AA) != 0;
    // everything optional goes to the FULL variants
    // colour with per-view faces (NR_VIEW_FACES) also takes the full variants: only they add the view's row offset to
    // faces_textures, which costs the plain colour variant (config 2) spill traffic
    const bool full = a.lights.num > 0 || a.lights.backgrounds || a.wmap || a.dmap || !a.images || (a.R & 15) ||
                      (rgb && a.face_stride != 0);
    ProfScope p(PROF_RASTER, stream);
    if (a.flags & FLAG_FACE_TEX) {     // per-face texture cubes: colour, full-featured variants of their own
        const long long px = (long long)a.B * a.R * a.R;
        switch ((aa ? 1 : 0) | (a.fine ? 2 : 0)) {
            case 0: launch_after(1, px, k_raster<true, false, true, false, TEX_CUBE>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
            case 1: launch_after(1, px, k_raster<true, true, true, false, TEX_CUBE>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
            case 2: launch_after(1, px, k_raster<true, false, true, true, TEX_CUBE>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
            default: launch_after(1, px, k_raster<true, true, true, true, TEX_CUBE>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
        }
        return cudaGetLastError();
    }
    if (a.fine) {       // dense meshes: the full-featured kernels over 8x8 tiles
        switch ((rgb ? 1 : 0) | (aa ? 2 : 0)) {
            case 0: launch_after(1, (long long)a.B * a.R * a.R, k_raster<false, false, true, true>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
            case 1: launch_after(1, (long long)a.B * a.R * a.R, k_raster<true, false, true, true>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
            case 2: launch_after(1, (long long)a.B * a.R * a.R, k_raster<false, true, true, true>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
            default: launch_after(1, (long long)a.B * a.R * a.R, k_raster<true, true, true, true>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
        }
        return cudaGetLastError();
    }
    const int variant = (rgb ? 1 : 0) | (aa ? 2 : 0) | (full ? 4 : 0);
    switch (variant) {
        case 0: launch_after(1, (long long)a.B * a.R * a.R, k_raster<false, false, false, false>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
        case 1: launch_after(1, (long long)a.B * a.R * a.R, k_raster<true, false, false, false>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
        case 2: launch_after(1, (long long)a.B * a.R * a.R, k_raster<false, true, false, false>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
        case 3: launch_after(1, (long long)a.B * a.R * a.R, k_raster<true, true, false, false>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
        case 4: launch_after(1, (long long)a.B * a.R * a.R, k_raster<false, false, true, false>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
        case 5: launch_after(1, (long long)a.B * a.R * a.R, k_raster<true, false, true, false>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
        case 6: launch_after(1, (long long)a.B * a.R * a.R, k_raster<false, true, true, false>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
        default: launch_after(1, (long long)a.B * a.R * a.R, k_raster<true, true, true, false>, dim3(grid), dim3(TILE_THREADS), 0, stream, a); break;
    }
    return cudaGetLastError();
}

cudaError_t launch_weight_map_compat(const float *faces, const int32_t *fim, float *wmap, int B,
                                     int nf, int R, cudaStream_t stream) {
    const long long total = (long long)B * R * R;
    if (total <= 0) return cudaSuccess;
    ProfScope p(PROF_WEIGHT_MAP, stream);
    k_weight_map_compat<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(faces, fim, wmap, total, nf, R);
    return cudaGetLastError();
}

}  // namespace nr
