// nr_raster_zbuf.cu -- rasterizer for meshes of SMALL triangles (a 100 k-face sphere at 512^2, a million random
// triangles at 1024^2: hundreds of faces per 16x16 tile, a few pixels per face).
//
// There the tile pipeline (nr_binning.cu + nr_raster.cu) spends its time on the lists, not on pixels: tens of
// millions of (tile, face) pairs to count, scatter and sort into ascending face order, and a raster kernel that
// evaluates every face of a list for all 32 pixels of a warp block although the face covers a handful.  This
// path has NO lists and NO per-face records.  It turns the loops around:
//
//   k_zb_faces    one THREAD per (view, face): gathers the 3 vertices (rasterize.py:232), applies the tests that
//                 do not depend on the pixel (back-face :100-104, degenerate :118-121), finds the exact pixel box
//                 (:94-97), walks its pixels, evaluates the reference's edge functions (:107-116) and, where the
//                 pixel is covered, merges (cheap depth, face) into a 64-bit z-buffer in global memory with ONE
//                 atomicMin.  A face whose box is larger than ZB_BIG_AREA pixels is walked by its whole warp.
//   k_zb_slots    numbers the CONTESTED pixels (below) and hands each a list head.
//   k_zb_collect  one thread per (view, face) again: for the contested pixels inside its box (a few bit tests
//                 per row) the reference's own depth (:129-139) goes into that pixel's candidate list.
//   k_zb_resolve  one warp per contested pixel: orders its candidates by face index and replays the
//                 reference's sequential scan (:124-148) on them.
//   k_zb_shade    one CTA per 16x16 tile: winner -> weight map, texture sample, lights, silhouette, depth,
//                 flip, anti-aliasing (shade_block, nr_shade.cuh), and the backward's list of non-empty tiles.
//
// Why the minimum is enough.  The reference's z-test is a SEQUENTIAL scan with a 1e-4 hysteresis (:145-148), not
// a minimum.  But a candidate is only ever replaced by one at least delta closer, and the closest one is accepted
// whenever it arrives: for a pixel whose closest candidate is closer than every other by more than the
// hysteresis (plus the error bound of the cheap depth), the scan ends on that candidate whatever the order.
// atomicMin returns the minimum of the moment; a candidate that comes within the band of it marks the pixel
// contested (of two near candidates the later one always sees the earlier one or something closer still, so no
// near-tie with the FINAL minimum is missed), and so does everything irregular: weights of mixed sign (the
// c2 == 0 quirk of :109,114), depths that are not ordinary positive numbers, a depth within the error bound of
// near or far.  Contested pixels - a fraction of a percent - are decided by the exact replay.  face_index_map is
// bit-identical to the tile pipeline's and to the reference's (tests: every parity case runs through both).
//
// If the candidate pool overflows (nrBinStats.overflow; the host grows it for the next call) the lists are
// unusable and every contested pixel is decided by the reference's own loop over ALL faces of its view, one warp
// per pixel: slow, exact.
#include "nr_shade.cuh"

namespace nr {

constexpr unsigned long long ZB_EMPTY = ~0ull;
constexpr int ZB_CAND = 128;        // candidates of one contested pixel sorted in shared memory (more: loop over all faces)
constexpr int ZB_THREADS = 256;

// Everything the per-pixel tests need of one face, in registers.
struct ZbFace {
    float x0, y0, z0, x1, y1, z1, x2, y2, z2;
    float dx10, dy10, dx21, dy21, dx02, dy02;       // x1-x0, y1-y0, x2-x1, y2-y1, x0-x2, y0-y2 (rounded once, like :107-116)
    float k0, k1, k2;                               // the pixel-independent half of the raw weights (:130-132)
    float iz0, iz1, iz2;
    bool zreg;
    int fid;
};

__device__ __forceinline__ void zb_face_from_record(const FaceRec &r, int fid, ZbFace &f) {
    f.x0 = r.q0.x; f.y0 = r.q0.y; f.z0 = r.q0.z; f.x1 = r.q0.w;
    f.y1 = r.q1.x; f.z1 = r.q1.y; f.x2 = r.q1.z; f.y2 = r.q1.w; f.z2 = r.q2.x;
    f.dx10 = __fsub_rn(f.x1, f.x0); f.dy10 = __fsub_rn(f.y1, f.y0);
    f.dx21 = __fsub_rn(f.x2, f.x1); f.dy21 = __fsub_rn(f.y2, f.y1);
    f.dx02 = __fsub_rn(f.x0, f.x2); f.dy02 = __fsub_rn(f.y0, f.y2);
    f.k0 = __fmaf_rn(f.x1, f.y2, -__fmul_rn(f.x2, f.y1));
    f.k1 = __fmaf_rn(f.x2, f.y0, -__fmul_rn(f.x0, f.y2));
    f.k2 = __fmaf_rn(f.x0, f.y1, -__fmul_rn(f.x1, f.y0));
    f.zreg = face_z_regular(f.z0, f.z1, f.z2);
    f.iz0 = fast_rcp(f.z0); f.iz1 = fast_rcp(f.z1); f.iz2 = fast_rcp(f.z2);
    f.fid = fid;
}

// :107-116.  rn(a - b) == -rn(b - a), so the deltas above give the reference's bits.
__device__ __forceinline__ bool zb_inside(const ZbFace &f, float xp, float yp) {
    const float c1 = __fmaf_rn(__fsub_rn(yp, f.y0), f.dx10, -__fmul_rn(f.dy10, __fsub_rn(xp, f.x0)));
    const float c2 = __fmaf_rn(__fsub_rn(yp, f.y1), f.dx21, -__fmul_rn(f.dy21, __fsub_rn(xp, f.x1)));
    const float c3 = __fmaf_rn(__fsub_rn(yp, f.y2), f.dx02, -__fmul_rn(f.dy02, __fsub_rn(xp, f.x2)));
    return !((__fmul_rn(c1, c2) < 0.f) | (__fmul_rn(c2, c3) < 0.f));
}

// raw_weights() (nr_common.cuh) from the precomputed halves: same operations, same bits
__device__ __forceinline__ void zb_weights(const ZbFace &f, float xp, float yp, float &w0, float &w1, float &w2) {
    w0 = __fadd_rn(__fmaf_rn(yp, f.dx21, __fmul_rn(xp, -f.dy21)), f.k0);
    w1 = __fadd_rn(__fmaf_rn(yp, f.dx02, __fmul_rn(xp, -f.dy02)), f.k1);
    w2 = __fadd_rn(__fmaf_rn(yp, f.dx10, __fmul_rn(xp, -f.dy10)), f.k2);
}

__device__ __forceinline__ void zb_flag(const RasterArgs &a, int b, int x, int y) {
    atomicOr(a.zb_bitmap + ((size_t)b * a.R + y) * a.zb_wpr + (x >> 5), 1u << (x & 31));
}

// One (face, pixel) candidate that passed the inside test, first half: its cheap depth.  Returns true when that
// depth goes into the z-buffer (zb_commit); an irregular candidate marks its pixel contested here, one that
// can never win is dropped.
__device__ __forceinline__ bool zb_prepare(const RasterArgs &a, const ZbFace &f, float xp, float yp, int b, int x, int y, float &zf) {
    float w0, w1, w2;
    zb_weights(f, xp, yp, w0, w1, w2);
    if (!(f.zreg && weights_one_sign(w0, w1, w2))) {
        zb_flag(a, b, x, y);                // irregular: the exact scan decides this pixel
        return false;
    }
    zf = fast_zp(w0, w1, w2, f.iz0, f.iz1, f.iz2);
    const float m = FAST_Z_REL * zf;
    // :140-142 rejects zp <= near and zp >= far; a depth in (far - delta, far) is valid but can never pass the
    // z-test against the initial minimum `far`, nor against a smaller one: it is irrelevant as well
    const float top = a.far_plane - a.delta;
    if (zf < a.near_plane - m || zf > top + m) return false;
    // (a NaN fails every comparison above and the one below: contested)
    if (!(zf > a.near_plane + m && zf < top - m && zf * 1e-6f < a.delta)) {
        zb_flag(a, b, x, y);
        return false;
    }
    return true;
}
// ... second half, after the atomicMin returned the minimum of the moment (`old`)
__device__ __forceinline__ void zb_check(const RasterArgs &a, float zf, unsigned long long old, int b, int x, int y) {
    if (old == ZB_EMPTY) return;
    const float zo = __uint_as_float((unsigned)(old >> 32));
    // within the hysteresis (plus both error bounds and the rounding of depth_min - delta) of the minimum of
    // this moment: order may matter
    if (fabsf(zf - zo) < a.delta + 2.5f * FAST_Z_REL * fmaxf(zf, zo)) zb_flag(a, b, x, y);
}
__device__ __forceinline__ unsigned long long zb_key(float zf, int fid) {
    return ((unsigned long long)__float_as_uint(zf) << 32) | (unsigned)fid;
}

// Face f of view b: record + exact pixel box; false when no pixel can accept it.
__device__ __forceinline__ bool zb_setup(const RasterArgs &a, int b, int f, ZbFace &F, int &xlo, int &xhi, int &ylo, int &yhi) {
    FaceRec r;
    const bool alive = make_face_record(a.verts + (size_t)b * a.nv * 3, a.faces + (size_t)b * a.face_stride, f, a.nv, a.R,
                                        (a.flags & FLAG_BACKSIDE) ? 1 : 0, r, xlo, xhi, ylo, yhi, a.hdr);
    if (alive) zb_face_from_record(r, f, F);
    return alive;
}

// ---------------------------------------------------------------------------------------------- pass 1
// A CTA owns 256 consecutive (view, face) pairs.  Their pixel boxes differ wildly (1 .. hundreds of pixels), so
// "one thread walks its own face" leaves most lanes idle.  Instead:
//   * the CTA's faces are ordered by the WIDTH of their pixel box (counting sort in shared memory) and the boxes
//     are laid end to end in that order (prefix sum of the box areas);
//   * every thread takes the same number of consecutive box pixels, rounded to whole ROWS, a row per round.
//     Neighbouring lanes hold rows of (almost) equal width, so the column loop of a round - inside test
//     (:107-116), coverage as a bit mask - runs with the warp's lanes in step;
//   * the covered pixels are compacted into the warp's ring in shared memory (one warp scan per round), and the
//     ring is drained 128 entries at a time, four per lane: four cheap depths, four atomicMin issued back to
//     back, then the four checks.  The atomicMin has to RETURN the old minimum, a round trip to L2 of about a
//     microsecond under load: the kernel lives on how many of them it keeps in flight.
constexpr int ZB_RING = 512;        // ring entries per warp: drained at 128, a round adds at most 32 lanes x 8 columns
constexpr int ZB_DRAIN = 128;
constexpr int ZB_COLS = 8;          // columns per round; wider rows take several rounds
constexpr int ZB_ROW_COST = 4;      // a row costs about as much as this many pixels on top of its own: the threads get equal COSTS
constexpr int ZB_HUGE = 4096;       // pixel boxes larger than this, or wider than 32 columns, are walked by a whole warp, unqueued
constexpr int ZB_F_IRREGULAR = 1;   // depths that are not ordinary positive numbers (face_z_regular)
constexpr int ZB_F_RANGE = 2;       // a depth of this face may come near `near` / `far`: per-pixel range tests

struct ZbFacesShared {
    // of the CTA's faces, at their position in width order:
    // v = x0 y0 x1 y1 x2 y2 | dx10 dy10 dx21 dy21 dx02 dy02 | k0 k1 k2 | iz0 iz1 iz2 (ZbFace)
    float v[18][ZB_THREADS];
    int box[ZB_THREADS];            // xlo | ylo << 16
    int wh[ZB_THREADS];             // width | height << 16 of the pixel box
    int pixbase[ZB_THREADS];        // index of pixel (xlo, ylo) of the face's view in the z-buffer
    int fid[ZB_THREADS];            // face | ZB_F_* << 29  (huge faces: the plain face index, see `view`)
    int view[ZB_THREADS];           // huge faces only
    int pre[ZB_THREADS + 1];        // exclusive prefix sum of the box costs (rows x (width + ZB_ROW_COST)) in width order (huge faces count 0)
    int start[ZB_THREADS + 1];      // first box pixel of every thread (a row boundary)
    int hist[40];                   // faces per width (0..31 = width - 1, 32 = huge), then their first positions
    int wsum[ZB_THREADS / 32];
    unsigned ring[ZB_THREADS / 32][ZB_RING];            // per warp: face position << 24 | row << 12 | column, inside the box
};
static_assert(sizeof(ZbFacesShared) <= 48 * 1024, "static shared memory");

// ... the whole face (huge faces)
__device__ __forceinline__ void zb_whole_face_from_shared(const ZbFacesShared &sh, int i, ZbFace &f) {
    f.dx10 = sh.v[6][i]; f.dy10 = sh.v[7][i]; f.dx21 = sh.v[8][i]; f.dy21 = sh.v[9][i]; f.dx02 = sh.v[10][i]; f.dy02 = sh.v[11][i];
    f.k0 = sh.v[12][i]; f.k1 = sh.v[13][i]; f.k2 = sh.v[14][i];
    f.iz0 = sh.v[15][i]; f.iz1 = sh.v[16][i]; f.iz2 = sh.v[17][i];
    f.zreg = (sh.fid[i] & (ZB_F_IRREGULAR << 29)) == 0;
    f.fid = sh.fid[i] & 0x1fffffff;
    f.x0 = sh.v[0][i]; f.y0 = sh.v[1][i]; f.x1 = sh.v[2][i]; f.y1 = sh.v[3][i]; f.x2 = sh.v[4][i]; f.y2 = sh.v[5][i];
    f.z0 = f.z1 = f.z2 = 0.f;       // (the cheap depth uses the reciprocals)
}

// contested-pixel flag from the z-buffer index of the pixel
__device__ __forceinline__ void zb_flag_pix(const RasterArgs &a, unsigned pix) {
    if ((a.R & 31) == 0) {
        atomicOr(a.zb_bitmap + (pix >> 5), 1u << (pix & 31));
    } else {
        const unsigned rowi = pix / (unsigned)a.R, x = pix - rowi * (unsigned)a.R;      // rowi = view * R + y
        atomicOr(a.zb_bitmap + (size_t)rowi * a.zb_wpr + (x >> 5), 1u << (x & 31));
    }
}

// Ring entries [head, head + n) of the warp (n <= 128): cheap depth, atomicMin, check; four per lane in flight.
template <bool POW2>
__device__ __forceinline__ void zb_drain(const RasterArgs &a, const ZbFacesShared &sh, const unsigned *ring, int head, int n, int lane,
                                         const PixGrid &grid) {
    const int R = a.R;
    float zf[4];
    unsigned pix[4];
    int fv[4];
    bool go[4];
    unsigned long long old[4];
    unsigned flags = 0u;                // contested pixels among my four
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int h = k * 32 + lane;
        go[k] = false;
        if (h < n) {
            const unsigned hc = ring[(head + h) & (ZB_RING - 1)];
            const int li = hc >> 24, col = (int)(hc & 0xfff), row = (int)((hc >> 12) & 0xfff);
            const int bx = sh.box[li];
            const int x = (bx & 0xffff) + col, y = (int)((unsigned)bx >> 16) + row;
            pix[k] = (unsigned)(sh.pixbase[li] + row * R + col);
            const int fl = sh.fid[li];
            fv[k] = fl & 0x1fffffff;
            const float xp = POW2 ? __fmul_rn((float)(2 * x + 1 - R), grid.invR) : pix_center(x, R);
            const float yp = POW2 ? __fmul_rn((float)(2 * y + 1 - R), grid.invR) : pix_center(y, R);
            // zb_weights() / zb_prepare() from the shared copy of the face
            const float w0 = __fadd_rn(__fmaf_rn(yp, sh.v[8][li], __fmul_rn(xp, -sh.v[9][li])), sh.v[12][li]);
            const float w1 = __fadd_rn(__fmaf_rn(yp, sh.v[10][li], __fmul_rn(xp, -sh.v[11][li])), sh.v[13][li]);
            const float w2 = __fadd_rn(__fmaf_rn(yp, sh.v[6][li], __fmul_rn(xp, -sh.v[7][li])), sh.v[14][li]);
            // weights_one_sign(), branch-free (a NaN weight makes the sum a NaN)
            const float ws = __fadd_rn(__fadd_rn(w0, w1), w2);
            const bool regular = ((fminf(w0, fminf(w1, w2)) >= 0.f) | (fmaxf(w0, fmaxf(w1, w2)) <= 0.f)) & (ws == ws) &
                                 ((fl & (ZB_F_IRREGULAR << 29)) == 0);
            zf[k] = fast_zp(w0, w1, w2, sh.v[15][li], sh.v[16][li], sh.v[17][li]);
            go[k] = regular;
            bool flag = !regular;               // irregular: the exact scan decides this pixel
            if (regular && (fl & (ZB_F_RANGE << 29))) {
                // (zb_prepare) :140-142 rejects zp <= near and zp >= far; a depth in (far - delta, far) is valid but can
                // never pass the z-test against the initial minimum `far`, nor against a smaller one
                const float m = FAST_Z_REL * zf[k], top = a.far_plane - a.delta;
                if (zf[k] < a.near_plane - m || zf[k] > top + m) go[k] = false;
                else if (!(zf[k] > a.near_plane + m && zf[k] < top - m && zf[k] * 1e-6f < a.delta)) {      // (NaN: contested)
                    go[k] = false;
                    flag = true;
                }
            }
            if (flag) flags |= 1u << k;
        }
    }
    if (__any_sync(0xffffffffu, flags != 0u)) {      // rare
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (flags & (1u << k)) zb_flag_pix(a, pix[k]);
        flags = 0u;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (go[k]) old[k] = atomicMin(a.zbuf + pix[k], zb_key(zf[k], fv[k]));
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (go[k] && old[k] != ZB_EMPTY) {
            // (zb_check) within the hysteresis (plus both error bounds and the rounding of depth_min - delta) of the
            // minimum of this moment: order may matter
            const float zo = __uint_as_float((unsigned)(old[k] >> 32));
            if (fabsf(zf[k] - zo) < a.delta + 2.5f * FAST_Z_REL * fmaxf(zf[k], zo)) flags |= 1u << k;
        }
    if (__any_sync(0xffffffffu, flags != 0u)) {      // rare
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (flags & (1u << k)) zb_flag_pix(a, pix[k]);
    }
}

// VIEW_FACES: faces [B, nf, 3] (NR_VIEW_FACES).  A variant of its own: the view's row offset in the variant
// for shared faces measured 0.7 % slower at config 4.
template <bool POW2, bool VIEW_FACES>
__global__ void __launch_bounds__(ZB_THREADS, 4)
k_zb_faces(const RasterArgs a) {
    pdl_trigger();      // (nr_kernels.h) the next pass may be scheduled as this one's CTAs leave
    __shared__ ZbFacesShared sh;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int R = a.R;
    const PixGrid grid(R);
    auto center = [&](int i) -> float { return POW2 ? __fmul_rn((float)(2 * i + 1 - R), grid.invR) : pix_center(i, R); };
    const long long idx = (long long)blockIdx.x * ZB_THREADS + tid;
    const bool in = idx < (long long)a.B * a.nf;
    const int b = in ? (int)(idx / a.nf) : 0, f = in ? (int)(idx % a.nf) : 0;
    if (tid < 40) sh.hist[tid] = 0;
    __syncthreads();
    // ---- per-face setup (rasterize.py:232, :94-104, :118-121)
    int key, rank;
    ZbFace F;
    int xlo = 1, xhi = 0, ylo = 1, yhi = 0;
    bool alive;
    {
        FaceRec r;
        alive = in && make_face_record(a.verts + (size_t)b * a.nv * 3, VIEW_FACES ? a.faces + (size_t)b * a.face_stride : a.faces,
                                       f, a.nv, R, (a.flags & FLAG_BACKSIDE) ? 1 : 0, r, xlo, xhi, ylo, yhi, a.hdr);
        // the exact pixel box for the collect pass, which then needs no vertices for faces that touch nothing contested
        if (in) a.zb_box[idx] = alive ? make_uint2((unsigned)xlo | ((unsigned)xhi << 16), (unsigned)ylo | ((unsigned)yhi << 16))
                                      : make_uint2(DEAD_BBOX, 0u);
        zb_face_from_record(r, f, F);
    }
    const int w = xhi - xlo + 1, h = yhi - ylo + 1;
    const bool huge = alive && (w * h > ZB_HUGE || w > 32);
    // ---- width order: position = first position of my width + my rank among the faces of that width
    key = huge ? 32 : w - 1;
    rank = alive ? atomicAdd(&sh.hist[key], 1) : 0;
    __syncthreads();
    if (wid == 0) {
        const int c = sh.hist[lane];
        int inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        const int nh = sh.hist[32];
        __syncwarp();
        sh.hist[lane] = inc - c;
        if (lane == 31) {
            sh.hist[32] = inc;              // number of faces that go through the rows = first position of the huge ones
            sh.hist[33] = inc + nh;         // live faces
        }
    }
    __syncthreads();
    const int n_rows = sh.hist[32], n_live = sh.hist[33];
    if (alive) {
        const int pos = sh.hist[key] + rank;
        sh.v[0][pos] = F.x0; sh.v[1][pos] = F.y0; sh.v[2][pos] = F.x1; sh.v[3][pos] = F.y1; sh.v[4][pos] = F.x2; sh.v[5][pos] = F.y2;
        sh.v[6][pos] = F.dx10; sh.v[7][pos] = F.dy10; sh.v[8][pos] = F.dx21; sh.v[9][pos] = F.dy21; sh.v[10][pos] = F.dx02; sh.v[11][pos] = F.dy02;
        sh.v[12][pos] = F.k0; sh.v[13][pos] = F.k1; sh.v[14][pos] = F.k2;
        sh.v[15][pos] = F.iz0; sh.v[16][pos] = F.iz1; sh.v[17][pos] = F.iz2;
        sh.box[pos] = xlo | (ylo << 16);
        sh.wh[pos] = w | (h << 16);
        sh.pixbase[pos] = (b * R + ylo) * R + xlo;
        // A regular face's cheap depths lie in [min z, max z] up to FAST_Z_REL (same-sign weights): when that interval
        // is clear of near and of far - delta by a wide margin, zb_prepare's range tests pass for every pixel
        const float zmin = fminf(F.z0, fminf(F.z1, F.z2)), zmax = fmaxf(F.z0, fmaxf(F.z1, F.z2));
        const float lo = zmin * (1.f - 8e-6f), hi = zmax * (1.f + 8e-6f), top = a.far_plane - a.delta;
        const float cmax = fmaxf(fmaxf(fmaxf(fabsf(F.x0), fabsf(F.x1)), fmaxf(fabsf(F.x2), fabsf(F.y0))), fmaxf(fabsf(F.y1), fabsf(F.y2)));
        const bool clear = F.zreg && lo > a.near_plane + 8e-6f * hi && hi < top - 8e-6f * hi && hi * 1.001e-6f < a.delta &&
                           cmax < 1e6f;         // (finite weights of ordinary size)
        sh.fid[pos] = f | (((F.zreg ? 0 : ZB_F_IRREGULAR) | (clear ? 0 : ZB_F_RANGE)) << 29);
        sh.view[pos] = b;
    }
    __syncthreads();
    // ---- the boxes end to end, in width order
    {
        const int wh_ = tid < n_rows ? sh.wh[tid] : 0;
        const int my = tid < n_rows ? ((wh_ & 0xffff) + ZB_ROW_COST) * (int)((unsigned)wh_ >> 16) : 0;
        int inc = my;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) sh.wsum[wid] = inc;
        __syncthreads();
        int base = 0;
#pragma unroll
        for (int k = 0; k < ZB_THREADS / 32; ++k)
            if (k < wid) base += sh.wsum[k];
        sh.pre[tid] = base + inc - my;
        if (tid == ZB_THREADS - 1) sh.pre[ZB_THREADS] = base + inc;
        __syncthreads();
    }
    const int total = sh.pre[ZB_THREADS];
    // ---- my share: `chunk` box pixels from the first row that starts at or behind pixel tid * chunk
    int p = 0, row = 0;
    {
        const int chunk = (total + ZB_THREADS - 1) / ZB_THREADS;
        const int t0 = min(tid * chunk, total);
        int st = total;
        if (t0 < total) {
            int lo = 0, hi = n_rows;                // first j with pre[j] > t0 (pre[n_rows] = total > t0)
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (sh.pre[mid] > t0) hi = mid; else lo = mid + 1;
            }
            p = lo - 1;
            const int wh_ = sh.wh[p], fw_ = (wh_ & 0xffff) + ZB_ROW_COST;
            row = (t0 - sh.pre[p] + fw_ - 1) / fw_;
            if (row == (int)((unsigned)wh_ >> 16)) {
                ++p;
                row = 0;
            }
            st = sh.pre[p] + row * (p < n_rows ? (sh.wh[p] & 0xffff) + ZB_ROW_COST : 0);
        }
        sh.start[tid] = st;
        if (tid == 0) sh.start[ZB_THREADS] = total;
        __syncthreads();
    }
    int rem = sh.start[tid + 1] - sh.start[tid];          // cost of this thread's rows
    // The warps run on their own from here.
    unsigned *ring = sh.ring[wid];
    const float step = 2.f * grid.invR;              // POW2: centre(i + 1) = centre(i) + 2 / R, exactly
    int head = 0, tail = 0;                                     // warp-uniform
    while (__any_sync(0xffffffffu, rem > 0)) {
        // ---- one row per lane
        const bool act = rem > 0;
        const int j = act ? p : 0;
        const int wh_ = sh.wh[j], bx = sh.box[j];
        const int fw = act ? (wh_ & 0xffff) : 0, fh = (int)((unsigned)wh_ >> 16);
        const int fx = bx & 0xffff, fy = (int)((unsigned)bx >> 16);
        const float x0 = sh.v[0][j], x1 = sh.v[2][j], x2 = sh.v[4][j];
        const float dx10 = sh.v[6][j], dy10 = sh.v[7][j], dx21 = sh.v[8][j], dy21 = sh.v[9][j], dx02 = sh.v[10][j], dy02 = sh.v[11][j];
        const float yp = center(fy + row);
        const float a1 = __fsub_rn(yp, sh.v[1][j]), a2 = __fsub_rn(yp, sh.v[3][j]), a3 = __fsub_rn(yp, sh.v[5][j]);
        const unsigned coderow = ((unsigned)j << 24) | ((unsigned)row << 12);
        const int wmax = __reduce_max_sync(0xffffffffu, fw);
        float xp = center(fx);
        for (int c0 = 0; c0 < wmax; c0 += ZB_COLS) {
            // inside tests (:107-116) over (at most) eight columns, coverage as a bit mask
            const int kend = min(ZB_COLS, wmax - c0);
            unsigned mask = 0u;               // bit (kend - 1 - k) = column c0 + k
#pragma unroll 2
            for (int k = 0; k < kend; ++k) {
                const float c1 = __fmaf_rn(a1, dx10, -__fmul_rn(dy10, __fsub_rn(xp, x0)));
                const float c2 = __fmaf_rn(a2, dx21, -__fmul_rn(dy21, __fsub_rn(xp, x1)));
                const float c3 = __fmaf_rn(a3, dx02, -__fmul_rn(dy02, __fsub_rn(xp, x2)));
                const bool hit = !((__fmul_rn(c1, c2) < 0.f) | (__fmul_rn(c2, c3) < 0.f));
                mask = mask + mask + (hit ? 1u : 0u);
                xp = POW2 ? __fadd_rn(xp, step) : center(fx + c0 + k + 1);
            }
            // columns beyond MY row (inactive lanes: all)
            const int over = c0 + kend - fw;
            if (over > 0) mask = over >= kend ? 0u : (mask >> over) << over;
            // exclusive scan of the hit counts over the lanes: where this lane's hits go
            const int cnt = __popc(mask);
            int inc = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += t;
            }
            int slot = tail + inc - cnt;
            const unsigned code = coderow + (unsigned)(c0 + kend - 1);
            while (mask) {
                ring[(slot++) & (ZB_RING - 1)] = code - (unsigned)(__ffs(mask) - 1);
                mask &= mask - 1;
            }
            tail += __shfl_sync(0xffffffffu, inc, 31);
            while (tail - head >= ZB_DRAIN) {
                __syncwarp();
                zb_drain<POW2>(a, sh, ring, head, ZB_DRAIN, lane, grid);
                __syncwarp();
                head += ZB_DRAIN;
            }
        }
        // ---- next row
        if (act) {
            rem -= fw + ZB_ROW_COST;
            if (++row == fh) {
                row = 0;
                ++p;
            }
        }
    }
    while (tail > head) {
        const int nd = min(tail - head, ZB_DRAIN);
        __syncwarp();
        zb_drain<POW2>(a, sh, ring, head, nd, lane, grid);
        head += nd;
    }
    // ---- huge faces: the whole warp walks the box of one face, a lane per pixel: the lanes form a (32 / wb) x wb
    // patch, wb = the box width rounded up to a power of two (32 at most), that steps over the box; two patches
    // per round keep two atomics per lane in flight.  Warp k takes the huge faces k, k + 8, ...
    for (int src = n_rows + wid; src < n_live; src += ZB_THREADS / 32) {
        ZbFace G;
        zb_whole_face_from_shared(sh, src, G);
        const int sb = sh.view[src], gx0 = sh.box[src] & 0xffff, gy0 = (int)((unsigned)sh.box[src] >> 16);
        const int gw = sh.wh[src] & 0xffff, gx1 = gx0 + gw - 1, gy1 = gy0 + (int)((unsigned)sh.wh[src] >> 16) - 1;
        int shf = 0;
        while ((1 << shf) < gw && shf < 5) ++shf;
        const int wb = 1 << shf, rows = 32 >> shf, lc = lane & (wb - 1), lr = lane >> shf;
        unsigned long long *zb = a.zbuf + (size_t)sb * R * R;
        for (int yb = gy0; yb <= gy1; yb += 2 * rows) {
            for (int xb = gx0; xb <= gx1; xb += wb) {
                const int x = xb + lc;
                float zf[2];
                int py[2];
                bool go[2];
                unsigned long long old[2];
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    py[k] = yb + k * rows + lr;
                    go[k] = false;
                    if (x <= gx1 && py[k] <= gy1) {
                        const float xq = center(x), yq = center(py[k]);
                        if (zb_inside(G, xq, yq)) go[k] = zb_prepare(a, G, xq, yq, sb, x, py[k], zf[k]);
                    }
                }
#pragma unroll
                for (int k = 0; k < 2; ++k)
                    if (go[k]) old[k] = atomicMin(zb + (size_t)py[k] * R + x, zb_key(zf[k], G.fid));
#pragma unroll
                for (int k = 0; k < 2; ++k)
                    if (go[k]) zb_check(a, zf[k], old[k], sb, x, py[k]);
            }
        }
    }
    // statistics for the host: a mesh with many such faces belongs to the tile pipeline
    if (tid == 0 && n_live > n_rows) atomicAdd(&a.hdr->max_tile_faces, n_live - n_rows);
}

// ---------------------------------------------------------------------------------------------- pass 2
// Every contested pixel gets a slot: its list head, and (in the face index map, which is not written before the
// shade pass) the way from the pixel to the slot.
__global__ void __launch_bounds__(ZB_THREADS)
k_zb_slots(const RasterArgs a, long long words) {
    pdl_wait();
    pdl_trigger();
    __shared__ int s_warp[ZB_THREADS / 32], s_base;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long idx = (long long)blockIdx.x * ZB_THREADS + threadIdx.x;
    if (idx == 0) {
#pragma unroll
        for (int k = 0; k < TILE_LIST_HDR; ++k) const_cast<int32_t *>(a.tile_list)[k] = 0;
    }
    unsigned w = idx < words ? a.zb_bitmap[idx] : 0u;
    if (!__syncthreads_or(w != 0u)) return;               // (most CTAs of most calls)
    // the CTA takes its slots with ONE atomic (tens of thousands of them on one address would queue up in L2)
    const int n = __popc(w);
    int inc = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
#pragma unroll
        for (int k = 0; k < ZB_THREADS / 32; ++k) {
            const int c = s_warp[k];
            s_warp[k] = tot;
            tot += c;
        }
        s_base = 0;
        if (tot) {
            s_base = atomicAdd(&a.hdr->zb_slots, tot);
            atomicAdd(&a.hdr->total_pairs, tot);          // reported to the host: contested pixels of this call
        }
    }
    __syncthreads();
    if (!w) return;
    int slot = s_base + s_warp[wid] + inc - n;
    const long long row = idx / a.zb_wpr;                 // = b * R + y
    const int xw = (int)(idx % a.zb_wpr) * 32;
    {
        // coarse bitmap: the OR of eight rows, so that the collect pass clears a face's box with a load or two
        const int b = (int)(row / a.R), y = (int)(row % a.R);
        atomicOr(a.zb_coarse + ((size_t)b * a.zb_crows + (y >> 3)) * a.zb_wpr + (idx % a.zb_wpr), w);
    }
    while (w) {
        const int x = xw + __ffs(w) - 1;
        w &= w - 1;
        const long long pix = row * a.R + x;
        if (slot < a.zb_slot_cap) {
            a.zb_pix_of[slot] = (int)pix;
            a.zb_head[slot] = -1;
            a.fim[pix] = slot;
        } else {
            a.fim[pix] = 0x7fffffff;
            a.hdr->overflow = 1;
        }
        ++slot;
    }
}

// ---------------------------------------------------------------------------------------------- pass 3
// The reference's own depth of face F at a contested pixel -> the pixel's candidate list.
__device__ __forceinline__ void zb_collect_pixel(const RasterArgs &a, const ZbFace &F, const PixGrid &grid, int b, int x, int y) {
    const float xp = grid.center(x), yp = grid.center(y);
    if (!zb_inside(F, xp, yp)) return;
    float w0, w1, w2;
    zb_weights(F, xp, yp, w0, w1, w2);
    const float zp = exact_zp(w0, w1, w2, F.z0, F.z1, F.z2);
    // :140-142; a NaN depth passes that test but then fails zp <= depth_min - delta: it never matters
    if (zp <= a.near_plane || a.far_plane <= zp || zp != zp) return;
    const int slot = a.fim[((size_t)b * a.R + y) * a.R + x];
    if (slot >= a.zb_slot_cap) return;                   // no slot: the overflow path decides this pixel
    const int node = atomicAdd(&a.hdr->zb_nodes, 1);
    if (node >= a.zb_node_cap) {
        a.hdr->overflow = 1;
        return;
    }
    // the scan skips a face when depth_min < z0 && depth_min < z1 && depth_min < z2 (:124-126): with a NaN corner
    // depth that is never true, otherwise it is depth_min < min(z)
    const float zc = (F.z0 != F.z0 || F.z1 != F.z1 || F.z2 != F.z2) ? -__int_as_float(0x7f800000) : fminf(F.z0, fminf(F.z1, F.z2));
    const int next = atomicExch(a.zb_head + slot, node);
    a.zb_nodes[node] = make_int4(F.fid, __float_as_int(zp), __float_as_int(zc), next);
}

constexpr int ZB_COLLECT_PER_THREAD = 4;        // faces per thread: four box loads (and the coarse lookups behind them) in flight
constexpr int ZB_COLLECT_FACES = ZB_THREADS * ZB_COLLECT_PER_THREAD;
constexpr int ZB_PAIR_CAP = 2048;               // (face, contested pixel) pairs of a CTA gathered in shared memory; more are taken one by one

// Face f of view b for the exact depth: its vertices and what zb_inside / zb_weights need.  The face-level tests
// were k_zb_faces' business: only faces with a live pixel box get here.
__device__ __forceinline__ void zb_gather(const RasterArgs &a, int b, int f, ZbFace &F) {
    int i0 = 3 * f, i1 = 3 * f + 1, i2 = 3 * f + 2;
    if (a.faces) {
        const int32_t *fr = a.faces + (size_t)b * a.face_stride + 3 * (size_t)f;
        i0 = __ldg(fr); i1 = __ldg(fr + 1); i2 = __ldg(fr + 2);
    }
    const float *vb = a.verts + (size_t)b * a.nv * 3;
    FaceRec r;
    r.q0 = make_float4(__ldg(vb + 3 * (size_t)i0), __ldg(vb + 3 * (size_t)i0 + 1), __ldg(vb + 3 * (size_t)i0 + 2), __ldg(vb + 3 * (size_t)i1));
    r.q1 = make_float4(__ldg(vb + 3 * (size_t)i1 + 1), __ldg(vb + 3 * (size_t)i1 + 2), __ldg(vb + 3 * (size_t)i2), __ldg(vb + 3 * (size_t)i2 + 1));
    r.q2 = make_float4(__ldg(vb + 3 * (size_t)i2 + 2), 0.f, 0.f, 0.f);
    zb_face_from_record(r, f, F);
}

// Three steps, each on full warps: (1) a thread per face: pixel box (as pass 1 found it) against the coarse
// bitmap - most faces touch no contested pixel; (2) EIGHT lanes per face that passed, a row of its box each,
// against the bitmap itself: every contested pixel inside the box becomes a (face, pixel) pair; (3) a thread per
// pair: vertices, inside test, the reference's depth, the pixel's list.
__global__ void __launch_bounds__(ZB_THREADS)
k_zb_collect(const RasterArgs a) {
    __shared__ int s_queue[ZB_COLLECT_FACES];
    __shared__ uint2 s_qbox[ZB_COLLECT_FACES];
    __shared__ int2 s_pairs[ZB_PAIR_CAP];
    __shared__ int s_n, s_np;
    pdl_wait();
    pdl_trigger();
    if (a.hdr->zb_slots == 0) return;                     // nothing contested (uniform over the grid)
    const int tid = threadIdx.x, lane = tid & 31;
    const long long total = (long long)a.B * a.nf;
    const long long cta0 = (long long)blockIdx.x * ZB_COLLECT_FACES;
    const int b0 = (int)(cta0 / a.nf);                    // view of the CTA's first face
    const unsigned f0 = (unsigned)(cta0 - (long long)b0 * a.nf);
    const bool two_views = a.nf >= ZB_COLLECT_FACES;      // the CTA's faces belong to at most two views
    auto view_face = [&](int slot, int &b, int &f) {      // slot = position in the CTA's range of (view, face) pairs
        const unsigned o = f0 + (unsigned)slot;
        const unsigned q = two_views ? (o >= (unsigned)a.nf ? 1u : 0u) : o / (unsigned)a.nf;
        b = b0 + (int)q;
        f = (int)(o - q * (unsigned)a.nf);
    };
    const PixGrid grid(a.R);
    // A box of at most 32 columns [c0, c1] lies in bitmap words w0 = c0 >> 5 and (perhaps) w0 + 1: its bits there
    auto word_masks = [](int c0, int c1, unsigned &m0, unsigned &m1) {
        const int w0 = c0 >> 5;
        m0 = 0xffffffffu << (c0 & 31);
        m1 = 0u;
        if ((c1 >> 5) == w0) m0 &= 0xffffffffu >> (31 - (c1 & 31));
        else m1 = 0xffffffffu >> (31 - (c1 & 31));
    };
    if (tid == 0) {
        s_n = 0;
        s_np = 0;
    }
    __syncthreads();
    // ---- (1) the faces' pixel boxes as pass 1 found them, against the coarse bitmap
    uint2 box[ZB_COLLECT_PER_THREAD];
#pragma unroll
    for (int k = 0; k < ZB_COLLECT_PER_THREAD; ++k) {
        const long long idx = cta0 + k * ZB_THREADS + tid;
        box[k] = idx < total ? __ldg(a.zb_box + idx) : make_uint2(DEAD_BBOX, 0u);
    }
    unsigned huge_mask[ZB_COLLECT_PER_THREAD];
#pragma unroll
    for (int k = 0; k < ZB_COLLECT_PER_THREAD; ++k) {
        const int xlo = (int)(box[k].x & 0xffff), xhi = (int)(box[k].x >> 16), ylo = (int)(box[k].y & 0xffff), yhi = (int)(box[k].y >> 16);
        const bool alive = xlo <= xhi;
        const bool huge = alive && ((xhi - xlo + 1) * (yhi - ylo + 1) > ZB_HUGE || xhi - xlo + 1 > 32);
        huge_mask[k] = __ballot_sync(0xffffffffu, huge);
        if (alive && !huge) {
            int b, f;
            view_face(k * ZB_THREADS + tid, b, f);
            unsigned m0, m1;
            word_masks(xlo, xhi, m0, m1);
            const unsigned *cb = a.zb_coarse + ((size_t)b * a.zb_crows + (ylo >> 3)) * a.zb_wpr + (xlo >> 5);
            unsigned any = 0u;
            for (int cy = ylo >> 3; cy <= (yhi >> 3); ++cy, cb += a.zb_wpr) {
                any |= __ldg(cb) & m0;
                if (m1) any |= __ldg(cb + 1) & m1;
            }
            if (any) {
                const int q = atomicAdd(&s_n, 1);
                s_queue[q] = k * ZB_THREADS + tid;
                s_qbox[q] = box[k];
            }
        }
    }
    __syncthreads();
    // ---- (2) the rows of the boxes that passed: lane group g of 8 takes face g, g + 32, ..., its lanes the rows
    const int nq = s_n;
#ifdef NR_ZB_STATS
    if (tid == 0) atomicAdd(&a.hdr->zb_work[1], nq);
#endif
    for (int q = tid >> 3; q < nq; q += ZB_THREADS / 8) {
        const int slot = s_queue[q];
        const uint2 bx = s_qbox[q];
        const int qx0 = (int)(bx.x & 0xffff), qx1 = (int)(bx.x >> 16), qy0 = (int)(bx.y & 0xffff), qy1 = (int)(bx.y >> 16);
        int qb, qf;
        view_face(slot, qb, qf);
        unsigned m0, m1;
        word_masks(qx0, qx1, m0, m1);
        const int w0 = qx0 >> 5;
        const unsigned *bm = a.zb_bitmap + (size_t)qb * a.R * a.zb_wpr + w0;
        for (int y = qy0 + (tid & 7); y <= qy1; y += 8) {
            const unsigned *rowp = bm + (size_t)y * a.zb_wpr;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (h == 1 && !m1) break;
                unsigned bits = __ldg(rowp + h) & (h ? m1 : m0);
                while (bits) {
                    const int x = (w0 + h) * 32 + __ffs(bits) - 1;
                    bits &= bits - 1;
                    const int n = atomicAdd(&s_np, 1);
                    if (n < ZB_PAIR_CAP) {
                        s_pairs[n] = make_int2(slot, x | (y << 16));
                    } else {                              // (a CTA whose faces sit on thousands of contested pixels)
                        ZbFace F;
                        zb_gather(a, qb, qf, F);
                        zb_collect_pixel(a, F, grid, qb, x, y);
                    }
                }
            }
        }
    }
    __syncthreads();
    // ---- (3) the pairs
    const int np = min(s_np, ZB_PAIR_CAP);
#ifdef NR_ZB_STATS
    if (tid == 0) atomicAdd(&a.hdr->zb_work[2], s_np);
#endif
    for (int i = tid; i < np; i += ZB_THREADS) {
        const int2 pr = s_pairs[i];
        int pb, pf;
        view_face(pr.x, pb, pf);
        ZbFace F;
        zb_gather(a, pb, pf, F);
        zb_collect_pixel(a, F, grid, pb, pr.y & 0xffff, pr.y >> 16);
    }
    auto col_mask = [](int wq, int c0, int c1) -> unsigned {
        const int lo = max(c0 - wq * 32, 0), hi = min(c1 - wq * 32, 31);
        return (0xffffffffu >> (31 - hi)) & (0xffffffffu << lo);
    };
    // huge faces: the whole warp, a lane per (row, word)
#pragma unroll
    for (int k = 0; k < ZB_COLLECT_PER_THREAD; ++k) {
        unsigned todo = huge_mask[k];
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            int sb, sf;
            view_face(k * ZB_THREADS + (tid & ~31) + src, sb, sf);
            ZbFace G;
            int gx0, gx1, gy0, gy1;
            if (!zb_setup(a, sb, sf, G, gx0, gx1, gy0, gy1)) continue;
            const int w0 = gx0 >> 5, nw = (gx1 >> 5) - w0 + 1;
            const int items = nw * (gy1 - gy0 + 1);           // (row, word) pairs, a lane each
            for (int j = lane; j < items; j += 32) {
                const int y = gy0 + j / nw, wq = w0 + j % nw;
                unsigned bits = __ldg(a.zb_bitmap + ((size_t)sb * a.R + y) * a.zb_wpr + wq) & col_mask(wq, gx0, gx1);
                while (bits) {
                    const int x = wq * 32 + __ffs(bits) - 1;
                    bits &= bits - 1;
                    zb_collect_pixel(a, G, grid, sb, x, y);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------- pass 4
// The reference's loop (:82-149) for ONE pixel over all faces of its view, by a warp (overflow path, and pixels
// with more candidates than ZB_CAND).  Returns the winning face or -1.
__device__ __noinline__ int zb_scan_all_faces(const RasterArgs &a, int b, float xp, float yp, int lane) {
    const float *vb = a.verts + (size_t)b * a.nv * 3;
    const bool cull = !(a.flags & FLAG_BACKSIDE);
    float depth_min = a.far_plane;
    int best = -1;
    for (int g = 0; g < a.nf; g += 32) {
        const int f = g + lane;
        float zp = 0.f, zc = 0.f;
        bool keep = false;
        if (f < a.nf) {
            int i0 = 3 * f, i1 = 3 * f + 1, i2 = 3 * f + 2;
            if (a.faces) {
                const int32_t *fr = a.faces + (size_t)b * a.face_stride + 3 * (size_t)f;
                i0 = __ldg(fr); i1 = __ldg(fr + 1); i2 = __ldg(fr + 2);
            }
            if ((unsigned)i0 < (unsigned)a.nv && (unsigned)i1 < (unsigned)a.nv && (unsigned)i2 < (unsigned)a.nv) {
                const float x0 = vb[3 * (size_t)i0], y0 = vb[3 * (size_t)i0 + 1], z0 = vb[3 * (size_t)i0 + 2];
                const float x1 = vb[3 * (size_t)i1], y1 = vb[3 * (size_t)i1 + 1], z1 = vb[3 * (size_t)i1 + 2];
                const float x2 = vb[3 * (size_t)i2], y2 = vb[3 * (size_t)i2 + 1], z2 = vb[3 * (size_t)i2 + 2];
                // :94-97 (a NaN coordinate fails no comparison here but yields a NaN depth below)
                keep = !(xp < fminf(x0, fminf(x1, x2)) || fmaxf(x0, fmaxf(x1, x2)) < xp || yp < fminf(y0, fminf(y1, y2)) ||
                         fmaxf(y0, fmaxf(y1, y2)) < yp);
                keep = keep && isfinite(x0) && isfinite(x1) && isfinite(x2) && isfinite(y0) && isfinite(y1) && isfinite(y2);
                // :100-104
                if (keep && cull && __fmul_rn(__fsub_rn(y2, y0), __fsub_rn(x1, x0)) > __fmul_rn(__fsub_rn(y1, y0), __fsub_rn(x2, x0))) keep = false;
                if (keep) {
                    // :107-116
                    const float c1 = __fmaf_rn(__fsub_rn(yp, y0), __fsub_rn(x1, x0), -__fmul_rn(__fsub_rn(y1, y0), __fsub_rn(xp, x0)));
                    const float c2 = __fmaf_rn(__fsub_rn(yp, y1), __fsub_rn(x2, x1), -__fmul_rn(__fsub_rn(y2, y1), __fsub_rn(xp, x1)));
                    const float c3 = __fmaf_rn(__fsub_rn(yp, y2), __fsub_rn(x0, x2), -__fmul_rn(__fsub_rn(y0, y2), __fsub_rn(xp, x2)));
                    keep = !((__fmul_rn(c1, c2) < 0.f) | (__fmul_rn(c2, c3) < 0.f));
                }
                if (keep) {
                    // :118-121
                    const float det = __fmaf_rn(x1, __fsub_rn(y2, y0), __fmaf_rn(x2, __fsub_rn(y0, y1), __fmul_rn(x0, __fsub_rn(y1, y2))));
                    keep = !((double)fabsf(det) < 0.00000001);
                }
                if (keep) {
                    float w0, w1, w2;
                    raw_weights(xp, yp, x0, y0, x1, y1, x2, y2, w0, w1, w2);
                    zp = exact_zp(w0, w1, w2, z0, z1, z2);
                    zc = (z0 != z0 || z1 != z1 || z2 != z2) ? -__int_as_float(0x7f800000) : fminf(z0, fminf(z1, z2));
                    keep = !(zp <= a.near_plane || a.far_plane <= zp) && zp == zp;
                }
            }
        }
        unsigned m = __ballot_sync(0xffffffffu, keep);
        while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            const float szp = __shfl_sync(0xffffffffu, zp, src), szc = __shfl_sync(0xffffffffu, zc, src);
            if (depth_min < szc) continue;                              // :124-126
            if (szp <= __fsub_rn(depth_min, a.delta)) {                  // :145-148
                depth_min = szp;
                best = g + src;
            }
        }
    }
    return best;
}

struct ZbResolveShared {
    int f[ZB_THREADS / 32][2][ZB_CAND];
    float z[ZB_THREADS / 32][2][ZB_CAND];
    float c[ZB_THREADS / 32][2][ZB_CAND];
};

__global__ void __launch_bounds__(ZB_THREADS)
k_zb_resolve(const RasterArgs a, long long words) {
    pdl_wait();
    pdl_trigger();
    __shared__ ZbResolveShared sh;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const PixGrid grid(a.R);
    const long long gw = (long long)blockIdx.x * (ZB_THREADS / 32) + wid, nwarps = (long long)gridDim.x * (ZB_THREADS / 32);
    const long long plane = (long long)a.R * a.R;
    auto put = [&](long long pix, int best) {
        if (lane == 0) a.zbuf[pix] = best >= 0 ? (unsigned long long)(unsigned)best : ZB_EMPTY;
    };
    if (a.hdr->overflow) {
        // lists unusable: every contested pixel by the loop over all faces
        for (long long wi = gw; wi < words; wi += nwarps) {
            unsigned bits = a.zb_bitmap[wi];
            const long long row = wi / a.zb_wpr;
            const int xw = (int)(wi % a.zb_wpr) * 32, b = (int)(row / a.R), y = (int)(row % a.R);
            while (bits) {
                const int x = xw + __ffs(bits) - 1;
                bits &= bits - 1;
                put(row * a.R + x, zb_scan_all_faces(a, b, grid.center(x), grid.center(y), lane));
            }
        }
        return;
    }
    const int slots = min(a.hdr->zb_slots, a.zb_slot_cap);
    int *cf = sh.f[wid][0], *sf = sh.f[wid][1];
    float *cz = sh.z[wid][0], *sz = sh.z[wid][1], *cc = sh.c[wid][0], *sc = sh.c[wid][1];
    for (long long slot = gw; slot < slots; slot += nwarps) {
        const long long pix = a.zb_pix_of[slot];
        // ---- the list into shared memory (lane 0 walks it)
        int count = 0;
        if (lane == 0) {
            for (int node = a.zb_head[slot]; node >= 0;) {
                const int4 nd = a.zb_nodes[node];
                if (count < ZB_CAND) {
                    cf[count] = nd.x;
                    cz[count] = __int_as_float(nd.y);
                    cc[count] = __int_as_float(nd.z);
                }
                ++count;
                node = nd.w;
            }
        }
        count = __shfl_sync(0xffffffffu, count, 0);
        __syncwarp();
        if (count > ZB_CAND) {
            const int b = (int)(pix / plane), rem = (int)(pix % plane);
            put(pix, zb_scan_all_faces(a, b, grid.center(rem % a.R), grid.center(rem / a.R), lane));
            continue;
        }
        // ---- order by face index (rank = number of smaller ids; ids are distinct), then the reference's scan
        for (int i = lane; i < count; i += 32) {
            const int fi = cf[i];
            int r = 0;
            for (int j = 0; j < count; ++j) r += cf[j] < fi;
            sf[r] = fi;
            sz[r] = cz[i];
            sc[r] = cc[i];
        }
        __syncwarp();
        float depth_min = a.far_plane;
        int best = -1;
        if (lane == 0) {
            for (int j = 0; j < count; ++j) {
                const float zp = sz[j];
                if (depth_min < sc[j]) continue;                         // :124-126
                if (zp <= __fsub_rn(depth_min, a.delta)) {                // :145-148
                    depth_min = zp;
                    best = sf[j];
                }
            }
        }
        put(pix, best);
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------- pass 5
template <bool RGB, bool AA, bool FULL>
__global__ void __launch_bounds__(TILE_THREADS)
k_zb_shade(const RasterArgs a) {
    pdl_wait();
    pdl_trigger();      // the backward
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int R = a.R;
    const PixGrid grid(R);
    const bool has_bg = FULL && RGB && a.lights.backgrounds != nullptr;
    // the caller's zero buffers (gradient accumulators of the coming backward) ride along: stores only
    const FillPlan plan = make_fill_plan(a);
    for (int fi = plan.all_tiles + blockIdx.x * (TILE_THREADS / 32) + wid; fi < plan.fill_items; fi += gridDim.x * (TILE_THREADS / 32))
        do_fill_item<AA, FULL, false>(a, plan, fi, lane);

    const int nt = a.ntx * a.ntx;
    const int b = blockIdx.x / nt, t = blockIdx.x % nt, ty = t / a.ntx, tx = t % a.ntx;
    int px, py;
    tile_pixel(tid, px, py);
    const int xi = tx * TILE + px, yi = ty * TILE + py;
    const bool valid = xi < R && yi < R;
    int best = -1;
    if (valid) {
        const unsigned long long key = a.zbuf[((size_t)b * R + yi) * R + xi];
        if (key != ZB_EMPTY) best = (int)(unsigned)(key & 0xffffffffu);
    }
    float bw0 = 0.f, bw1 = 0.f, bw2 = 0.f, bz0 = 0.f, bz1 = 0.f, bz2 = 0.f;
    // a plain silhouette needs the winner, not its weights: no vertex gather then (three dependent loads less)
    const bool need_weights = RGB || FULL || (a.flags & FLAG_DEPTH) || a.aux != nullptr;
    if (best >= 0 && need_weights) {
        int i0 = 3 * best, i1 = 3 * best + 1, i2 = 3 * best + 2;
        if (a.faces) {
            const int32_t *fr = a.faces + (size_t)b * a.face_stride + 3 * (size_t)best;
            i0 = __ldg(fr); i1 = __ldg(fr + 1); i2 = __ldg(fr + 2);
        }
        const float *vb = a.verts + (size_t)b * a.nv * 3;
        const float x0 = __ldg(vb + 3 * (size_t)i0), y0 = __ldg(vb + 3 * (size_t)i0 + 1);
        const float x1 = __ldg(vb + 3 * (size_t)i1), y1 = __ldg(vb + 3 * (size_t)i1 + 1);
        const float x2 = __ldg(vb + 3 * (size_t)i2), y2 = __ldg(vb + 3 * (size_t)i2 + 1);
        bz0 = __ldg(vb + 3 * (size_t)i0 + 2); bz1 = __ldg(vb + 3 * (size_t)i1 + 2); bz2 = __ldg(vb + 3 * (size_t)i2 + 2);
        raw_weights(grid.center(xi), grid.center(yi), x0, y0, x1, y1, x2, y2, bw0, bw1, bw2);
    }
    shade_block<RGB, AA, FULL>(a, b, xi, yi, valid, best, bw0, bw1, bw2, bz0, bz1, bz2, has_bg);
    // the backward walks the non-empty tiles only
    const int any = __syncthreads_or(best >= 0);
    if (any && tid == 0) {
        int32_t *tl = const_cast<int32_t *>(a.tile_list);
        const int i = atomicAdd(tl, 1);           // all in class 0
        reinterpret_cast<int4 *>(tl + TILE_LIST_HDR)[i] = make_int4(b, tx | (ty << 16), 0, 0);
    }
}

cudaError_t launch_raster_zbuf(const RasterArgs &a, cudaStream_t stream) {
    if (a.B <= 0 || a.R <= 0) return cudaSuccess;
    const long long faces = (long long)a.B * a.nf, words = (long long)a.B * a.R * a.zb_wpr;
    const long long plane = (long long)a.B * a.R * a.R;
    cudaError_t e;
    {
        ProfScope p(PROF_MEMSET, stream);
        // header, bitmap and coarse bitmap are adjacent
        const size_t coarse_words = (size_t)a.B * a.zb_crows * a.zb_wpr;
        if ((e = cudaMemsetAsync(a.hdr, 0, sizeof(BinHeader) + ((size_t)words + coarse_words) * sizeof(unsigned), stream)) != cudaSuccess) return e;
        if ((e = cudaMemsetAsync(a.zbuf, 0xff, (size_t)plane * sizeof(unsigned long long), stream)) != cudaSuccess) return e;
    }
    const unsigned face_ctas = (unsigned)((faces + ZB_THREADS - 1) / ZB_THREADS);
    if (face_ctas) {
        ProfScope p(PROF_ZB_FACES, stream);
        const bool pow2 = (a.R & (a.R - 1)) == 0;
        if (a.face_stride) {
            if (pow2) k_zb_faces<true, true><<<face_ctas, ZB_THREADS, 0, stream>>>(a);
            else k_zb_faces<false, true><<<face_ctas, ZB_THREADS, 0, stream>>>(a);
        } else {
            if (pow2) k_zb_faces<true, false><<<face_ctas, ZB_THREADS, 0, stream>>>(a);
            else k_zb_faces<false, false><<<face_ctas, ZB_THREADS, 0, stream>>>(a);
        }
    }
    {
        ProfScope p(PROF_ZB_RESOLVE, stream);
        launch_after(4, (long long)a.B * a.R * a.R, k_zb_slots, dim3((unsigned)((words + ZB_THREADS - 1) / ZB_THREADS)), dim3(ZB_THREADS), 0, stream, a, words);
        if (face_ctas)
            launch_after(4, (long long)a.B * a.R * a.R, k_zb_collect, dim3((unsigned)((faces + ZB_COLLECT_FACES - 1) / ZB_COLLECT_FACES)), dim3(ZB_THREADS), 0, stream, a);
        launch_after(4, (long long)a.B * a.R * a.R, k_zb_resolve, dim3(a.sm_count * 4), dim3(ZB_THREADS), 0, stream, a, words);
    }
    const bool rgb = (a.flags & FLAG_RGB) != 0, aa = (a.flags & FLAG_AA) != 0;
    const bool full = a.lights.num > 0 || a.lights.backgrounds || a.wmap || a.dmap || !a.images || (a.R & 15);
    const unsigned tiles = (unsigned)((long long)a.B * a.ntx * a.ntx);
    ProfScope p(PROF_ZB_SHADE, stream);
    // silhouettes of dense meshes are the measured case; everything else takes the full-featured variants
    if (!rgb && !aa && !full) launch_after(4, (long long)a.B * a.R * a.R, k_zb_shade<false, false, false>, dim3(tiles), dim3(TILE_THREADS), 0, stream, a);
    else if (rgb && aa) launch_after(4, (long long)a.B * a.R * a.R, k_zb_shade<true, true, true>, dim3(tiles), dim3(TILE_THREADS), 0, stream, a);
    else if (rgb) launch_after(4, (long long)a.B * a.R * a.R, k_zb_shade<true, false, true>, dim3(tiles), dim3(TILE_THREADS), 0, stream, a);
    else if (aa) launch_after(4, (long long)a.B * a.R * a.R, k_zb_shade<false, true, true>, dim3(tiles), dim3(TILE_THREADS), 0, stream, a);
    else launch_after(4, (long long)a.B * a.R * a.R, k_zb_shade<false, false, true>, dim3(tiles), dim3(TILE_THREADS), 0, stream, a);
    return cudaGetLastError();
}

}  // namespace nr
