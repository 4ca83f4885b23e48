// nr_binning.cu -- per-face setup and tile binning.
//
// Replaces the O(B * S^2 * nf) "every pixel scans every face" loop of the reference
// (rasterize_cuda_kernel.cu:82) by per-tile face lists.  The reference z-test is a
// SEQUENTIAL scan with a 1e-4 hysteresis (:145-148), so its result depends on the order
// faces are visited; every tile list is therefore delivered in ascending face index.
//
//   k_setup_count : one thread per (view, face). Gathers the 3 vertices (rasterize.py:232),
//                   applies the tests that do not depend on the pixel (back-face :100-104,
//                   degenerate :118-121), computes the EXACT set of pixel columns / rows whose
//                   centre passes the bounding-box test (:94-97), writes a 48-byte record and
//                   counts the face into every 16x16 tile its pixel box touches.
//   k_scan_tiles  : exclusive prefix sum of the per-tile counts (one CTA per view).
//   k_scatter     : writes face ids into the tile segments (slot order is arbitrary ...)
//   k_sort_tiles  : ... so every list is sorted in place: <= 256 ids by one warp in registers,
//                   <= 8192 by a CTA in shared memory, longer ones by a CTA in global memory.
#include <cooperative_groups.h>

#include "nr_kernels.h"

namespace nr {

__global__ void __launch_bounds__(256)
k_setup_count(const float *__restrict__ verts, const int32_t *__restrict__ faces, int face_stride, int B, int nv,
              int nf, int R, int draw_backside, FaceRec *__restrict__ rec,
              int *__restrict__ tile_count, int ntx, int tsh, BinHeader *__restrict__ hdr) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)B * nf) return;
    const int b = (int)(idx / nf), f = (int)(idx % nf);
    FaceRec r;
    int xlo, xhi, ylo, yhi;
    const bool alive = make_face_record(verts + (size_t)b * nv * 3, faces + (size_t)b * face_stride, f, nv, R, draw_backside, r,
                                        xlo, xhi, ylo, yhi, hdr);
    rec[idx] = r;
    if (!alive) return;

    int *tc = tile_count + (size_t)b * ntx * ntx;
    const int tx0 = xlo >> tsh, tx1 = xhi >> tsh, ty0 = ylo >> tsh, ty1 = yhi >> tsh;
    for (int ty = ty0; ty <= ty1; ++ty)
        for (int tx = tx0; tx <= tx1; ++tx) atomicAdd(&tc[ty * ntx + tx], 1);
}

// One CTA per view: exclusive scan of its tile counts; the view's base offset in the global
// pair list is claimed with one atomicAdd (segment placement is arbitrary, content is not).
__global__ void __launch_bounds__(1024)
k_scan_tiles(const int *__restrict__ tile_count, int *__restrict__ tile_offset,
             int *__restrict__ tile_cursor, int nt, int ntx, long long pair_capacity,
             BinHeader *__restrict__ hdr, int32_t *__restrict__ tile_list) {
    __shared__ int s_warp[32];
    __shared__ int s_base;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int *tc = tile_count + (size_t)b * nt;

    // pass 1: view total and longest list
    int sum = 0, mx = 0;
    for (int i = tid; i < nt; i += blockDim.x) {
        const int c = tc[i];
        sum += c;
        mx = max(mx, c);
    }
    for (int o = 16; o; o >>= 1) {
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0) s_warp[wid] = sum;
    if (lane == 0 && mx > 0) atomicMax(&hdr->max_tile_faces, mx);
    __syncthreads();
    if (tid == 0) {
        int tot = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += s_warp[w];
        const int base = atomicAdd(&hdr->total_pairs, tot);
        if ((long long)base + tot > pair_capacity) hdr->overflow = 1;
        s_base = base;
    }
    __syncthreads();
    int carry = s_base;
    __syncthreads();

    // pass 2: chunked block scan
    for (int c0 = 0; c0 < nt; c0 += blockDim.x) {
        const int i = c0 + tid;
        const int v = (i < nt) ? tc[i] : 0;
        int inc = v;
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) s_warp[wid] = inc;
        __syncthreads();
        if (wid == 0) {
            int w = s_warp[lane];
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += t;
            }
            s_warp[lane] = w;   // inclusive over warps
        }
        __syncthreads();
        const int warp_excl = (wid == 0) ? 0 : s_warp[wid - 1];
        const int excl = carry + warp_excl + inc - v;
        if (i < nt) {
            tile_offset[(size_t)b * nt + i] = excl;
            tile_cursor[(size_t)b * nt + i] = excl;
        }
        // append the non-empty tiles to the work list of their length class (one atomic per warp and class)
        const int cls = tile_class(v);
        const int cap = (int)gridDim.x * nt;
#pragma unroll
        for (int k = 0; k < TILE_CLASSES; ++k) {
            const unsigned busy = __ballot_sync(0xffffffffu, v > 0 && cls == k);
            if (busy) {
                int base = 0;
                if (lane == 0) base = atomicAdd(&tile_list[k], __popc(busy));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (v > 0 && cls == k) {
                    int4 *ent = reinterpret_cast<int4 *>(tile_list + TILE_LIST_HDR) + (size_t)k * cap + base +
                                __popc(busy & ((1u << lane) - 1u));
                    *ent = make_int4(b, (i % ntx) | ((i / ntx) << 16), excl, v);
                }
            }
        }
        carry += s_warp[31];
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256)
k_scatter(const FaceRec *__restrict__ rec, int B, int nf, int ntx, int tsh, int *__restrict__ tile_cursor,
          int32_t *__restrict__ pairs, long long pair_capacity, const BinHeader *__restrict__ hdr) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)B * nf) return;
    if (hdr->overflow) return;
    const float4 q2 = reinterpret_cast<const float4 *>(rec + idx)[2];
    const uint32_t bx = __float_as_uint(q2.y), by = __float_as_uint(q2.z);
    const int xlo = bx & 0xffff, xhi = bx >> 16;
    if (xlo > xhi) return;
    const int ylo = by & 0xffff, yhi = by >> 16;
    const int b = (int)(idx / nf), f = (int)(idx % nf);
    int *cur = tile_cursor + (size_t)b * ntx * ntx;
    const int tx0 = xlo >> tsh, tx1 = xhi >> tsh, ty0 = ylo >> tsh, ty1 = yhi >> tsh;
    for (int ty = ty0; ty <= ty1; ++ty)
        for (int tx = tx0; tx <= tx1; ++tx) {
            const int slot = atomicAdd(&cur[ty * ntx + tx], 1);
            if (slot < pair_capacity) pairs[slot] = f;
        }
}


// ---------------------------------------------------------------------------------------------------
// Small-mesh fast path: ONE kernel does all of the above.  A thread-block CLUSTER of 1..8 CTAs owns a
// view; CTA r of the cluster takes the r-th contiguous slice of the view's faces and keeps its tile
// counters, scans and (tile, face) pairs in its own shared memory:
//   A  face records (global) + per-tile counts of the slice (shared atomics)
//   -- cluster barrier --
//   B  every CTA reads the other slices' counts through distributed shared memory: a tile's list is
//      the concatenation of the slices' sub-lists in rank order (= ascending face index), so the
//      sub-list of slice r starts at  scan(total counts)[tile] + sum_{r' < r} count_{r'}[tile].
//      Rank 0 claims the view's segment of the global pair array (one atomicAdd) and writes the tile
//      counts and the heavy-first work-list entries.
//   -- cluster barrier (segment base) --
//   C  scatter of the slice's face ids into the shared pair array
//   D  per-tile ascending sort of the sub-lists (<= 128 ids: one warp, rank sort in registers; longer:
//      the whole CTA, counting rank sort in shared memory), written to their place in global memory
// Four dependent launches (~45 us at BASELINE config 2, all of it latency) become one.
// Taken when nf <= BINVIEW_MAX_FACES and tiles per view <= BINVIEW_MAX_TILES; a slice with more pairs
// than fit in shared memory raises hdr->overflow = 2: that call falls back to the all-faces scan in
// the raster kernel (exact), and the host uses the general path from then on.
constexpr int BINVIEW_THREADS = 1024;
constexpr int BINVIEW_MAX_FACES = 8192;
constexpr int BINVIEW_MAX_TILES = 4096;          // R <= 1024
constexpr int BINVIEW_PER = BINVIEW_MAX_TILES / BINVIEW_THREADS;
constexpr int BINVIEW_SMEM_PAIRS = 32768;
constexpr int BINVIEW_MAX_CLUSTER = 8;

// ascending sort of n <= 32 * G distinct ids read from src (shared), written to dst (global); one warp,
// rank sort with the ids in registers (position p lives in register p / 32 of lane p % 32)
template <int G>
__device__ __forceinline__ void warp_rank_sort(const int *src, int n, int32_t *dst, int lane) {
    int v[G], r[G];
#pragma unroll
    for (int k = 0; k < G; ++k) {
        v[k] = (k * 32 + lane < n) ? src[k * 32 + lane] : 0x7fffffff;
        r[k] = 0;
    }
#pragma unroll
    for (int kk = 0; kk < G; ++kk) {
        const int jn = min(32, n - 32 * kk);          // warp-uniform
        for (int j = 0; j < jn; ++j) {
            const int x = __shfl_sync(0xffffffffu, v[kk], j);
#pragma unroll
            for (int k = 0; k < G; ++k) r[k] += (x < v[k]);
        }
    }
#pragma unroll
    for (int k = 0; k < G; ++k)
        if (k * 32 + lane < n) dst[r[k]] = v[k];
}

__global__ void __launch_bounds__(BINVIEW_THREADS, 1)
k_bin_view(const float *__restrict__ verts, const int32_t *__restrict__ faces, int face_stride, int nv, int nf, int R,
           int draw_backside, int ntx, FaceRec *__restrict__ rec, int *__restrict__ tile_count,
           int32_t *__restrict__ pairs, long long pair_capacity, BinHeader *__restrict__ hdr,
           int32_t *__restrict__ tile_list) {
    namespace cg = cooperative_groups;
    pdl_trigger();      // the raster kernel may be scheduled as this kernel's CTAs leave (it waits for all of them)
    cg::cluster_group cluster = cg::this_cluster();
    const int cs = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    extern __shared__ int s_dyn[];
    const int nt = ntx * ntx;
    int *s_count = s_dyn;                 // [nt]   faces of this slice per tile
    int *s_cursor = s_dyn + nt;           // [nt]   position of the sub-list in s_pairs, then scatter cursor
    int *s_dst = s_dyn + 2 * nt;          // [nt]   position of the sub-list in the global pair array
    int *s_list = s_dyn + 3 * nt;         // [nt]   tiles with a sub-list (short ones from the front, long from the back)
    int *s_pairs = s_dyn + 4 * nt;        // [BINVIEW_SMEM_PAIRS]
    __shared__ int s_nlist, s_nlong, s_next;
    __shared__ int s_warp[32], s_warp_own[32];
    __shared__ int s_base, s_overflow;
    __shared__ int s_class_count[TILE_CLASSES], s_class_base[TILE_CLASSES];
    const int b = blockIdx.x / cs, views = gridDim.x / cs;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const float *vb = verts + (size_t)b * nv * 3;
    FaceRec *rec_b = rec + (size_t)b * nf;
    const int slice = ((nf + cs - 1) / cs + 31) & ~31;
    const int f_begin = min(nf, rank * slice), f_end = min(nf, f_begin + slice);

    for (int i = tid; i < nt; i += BINVIEW_THREADS) s_count[i] = 0;
    if (tid < TILE_CLASSES) s_class_count[tid] = 0;
    if (tid == 0) s_nlist = s_nlong = s_next = s_overflow = 0;
    __syncthreads();

    // ---- A: records and counts of this slice
    for (int f = f_begin + tid; f < f_end; f += BINVIEW_THREADS) {
        FaceRec r;
        int xlo, xhi, ylo, yhi;
        // (an int offset: b * 3 nf < 65536 * 3 * BINVIEW_MAX_FACES < 2^31, and no 64-bit pointer held across the kernel)
        const bool alive = make_face_record(vb, faces + b * face_stride, f, nv, R, draw_backside, r, xlo, xhi, ylo, yhi, hdr);
        rec_b[f] = r;
        if (!alive) continue;
        const int tx0 = xlo / TILE, tx1 = xhi / TILE, ty0 = ylo / TILE, ty1 = yhi / TILE;
        for (int ty = ty0; ty <= ty1; ++ty)
            for (int tx = tx0; tx <= tx1; ++tx) atomicAdd(&s_count[ty * ntx + tx], 1);
    }
    cluster.sync();

    // ---- B: scans (thread t owns tiles t * per .. t * per + per - 1)
    const int per = (nt + BINVIEW_THREADS - 1) / BINVIEW_THREADS;
    int own[BINVIEW_PER], tot[BINVIEW_PER], before[BINVIEW_PER];
    int sum_tot = 0, sum_own = 0, mx = 0;
#pragma unroll
    for (int k = 0; k < BINVIEW_PER; ++k) {
        const int i = tid * per + k;
        own[k] = tot[k] = before[k] = 0;
        if (k < per && i < nt) {
            own[k] = s_count[i];
            for (int r = 0; r < cs; ++r) {
                const int c = (r == rank) ? own[k] : cluster.map_shared_rank(s_count, r)[i];
                tot[k] += c;
                if (r < rank) before[k] += c;
            }
        }
        sum_tot += tot[k];
        sum_own += own[k];
        mx = max(mx, tot[k]);
    }
    int inc_tot = sum_tot, inc_own = sum_own;
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc_tot, o), u = __shfl_up_sync(0xffffffffu, inc_own, o);
        if (lane >= o) {
            inc_tot += t;
            inc_own += u;
        }
    }
    for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 31) {
        s_warp[wid] = inc_tot;
        s_warp_own[wid] = inc_own;
    }
    if (rank == 0 && lane == 0 && mx > 0) atomicMax(&hdr->max_tile_faces, mx);
    __syncthreads();
    if (wid == 0) {
        int w = s_warp[lane], u = s_warp_own[lane];
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, w, o), t2 = __shfl_up_sync(0xffffffffu, u, o);
            if (lane >= o) {
                w += t;
                u += t2;
            }
        }
        s_warp[lane] = w;     // inclusive over warps
        s_warp_own[lane] = u;
        if (lane == 31) {
            int ovf = 0;
            if (rank == 0) {
                const int base = atomicAdd(&hdr->total_pairs, w);
                if ((long long)base + w > pair_capacity) ovf = 1;
                s_base = base;
            }
            if (u > BINVIEW_SMEM_PAIRS) ovf = 2;
            if (ovf) {
                atomicMax(&hdr->overflow, ovf);
                s_overflow = ovf;
            }
        }
    }
    cluster.sync();
    const int base = *cluster.map_shared_rank(&s_base, 0);
    int excl_tot = (wid ? s_warp[wid - 1] : 0) + inc_tot - sum_tot;     // view-relative offset of this thread's first tile
    int excl_own = (wid ? s_warp_own[wid - 1] : 0) + inc_own - sum_own;
    const int excl_tot0 = excl_tot;
    int slot[BINVIEW_PER];
#pragma unroll
    for (int k = 0; k < BINVIEW_PER; ++k) {
        const int i = tid * per + k;
        slot[k] = -1;
        if (k < per && i < nt) {
            s_cursor[i] = excl_own;
            s_dst[i] = base + excl_tot + before[k];
            if (rank == 0) {
                tile_count[(size_t)b * nt + i] = tot[k];
                if (tot[k] > 0) slot[k] = atomicAdd(&s_class_count[tile_class(tot[k])], 1);
            }
            if (own[k] > 0) {
                // work list of phase D: short sub-lists (one warp each) from the front, long ones from the back
                if (own[k] <= 128) s_list[atomicAdd(&s_nlist, 1)] = i;
                else s_list[nt - 1 - atomicAdd(&s_nlong, 1)] = i;
            }
            excl_tot += tot[k];
            excl_own += own[k];
        }
    }
    __syncthreads();
    if (rank == 0) {
        if (tid < TILE_CLASSES) s_class_base[tid] = s_class_count[tid] ? atomicAdd(&tile_list[tid], s_class_count[tid]) : 0;
        __syncthreads();
        const int cap = views * nt;
        int off = excl_tot0;
#pragma unroll
        for (int k = 0; k < BINVIEW_PER; ++k) {
            const int i = tid * per + k;
            if (slot[k] >= 0) {
                const int c = tile_class(tot[k]);
                int4 *ent = reinterpret_cast<int4 *>(tile_list + TILE_LIST_HDR) + (size_t)c * cap + s_class_base[c] + slot[k];
                *ent = make_int4(b, (i % ntx) | ((i / ntx) << 16), base + off, tot[k]);
            }
            off += tot[k];
        }
    }
    // an overflow anywhere means the raster kernel scans all faces; the lists are not needed.  Every CTA
    // must outlive the remote reads of its shared memory, hence the barrier on both ways out.
    const bool skip = s_overflow != 0 || *cluster.map_shared_rank(&s_overflow, 0) != 0;
    if (!skip) {
        // ---- C: scatter into the shared pair array (slot order arbitrary)
        for (int f = f_begin + tid; f < f_end; f += BINVIEW_THREADS) {
            const float4 q2 = reinterpret_cast<const float4 *>(rec_b + f)[2];     // own write of phase A
            const uint32_t bx = __float_as_uint(q2.y), by = __float_as_uint(q2.z);
            const int xlo = bx & 0xffff, xhi = bx >> 16;
            if (xlo > xhi) continue;
            const int ylo = by & 0xffff, yhi = by >> 16;
            const int tx0 = xlo / TILE, tx1 = xhi / TILE, ty0 = ylo / TILE, ty1 = yhi / TILE;
            for (int ty = ty0; ty <= ty1; ++ty)
                for (int tx = tx0; tx <= tx1; ++tx) s_pairs[atomicAdd(&s_cursor[ty * ntx + tx], 1)] = f;
        }
        __syncthreads();

        // ---- D1: sub-lists of up to 128 ids, one warp per list, claimed dynamically
        const int nlist = s_nlist, nlong = s_nlong;
        while (true) {
            int j = 0;
            if (lane == 0) j = atomicAdd(&s_next, 1);
            j = __shfl_sync(0xffffffffu, j, 0);
            if (j >= nlist) break;
            const int i = s_list[j], n = s_count[i];
            const int *src = s_pairs + (s_cursor[i] - n);
            int32_t *dst = pairs + s_dst[i];
            if (n == 1) {
                if (lane == 0) dst[0] = src[0];
            } else if (n <= 32) {
                warp_rank_sort<1>(src, n, dst, lane);
            } else if (n <= 64) {
                warp_rank_sort<2>(src, n, dst, lane);
            } else {
                warp_rank_sort<4>(src, n, dst, lane);
            }
        }
        // ---- D2: longer sub-lists, the whole CTA per list: rank of every id by counting the smaller ones
        // (all threads read the same shared word at a time: broadcast, conflict-free)
        for (int l = 0; l < nlong; ++l) {
            const int i = s_list[nt - 1 - l], n = s_count[i];
            const int *src = s_pairs + (s_cursor[i] - n);
            int32_t *dst = pairs + s_dst[i];
            for (int e = tid; e < n; e += BINVIEW_THREADS) {
                const int v = src[e];
                int r = 0;
#pragma unroll 8
                for (int j = 0; j < n; ++j) r += (src[j] < v);
                dst[r] = v;
            }
        }
    }
    cluster.sync();
}

// Ascending in-place sort of every tile list of up to SMEM_SORT_CAP faces, grid-stride over the work
// list.  Lists that the scatter kernel happened to fill in face order only pay the sortedness check.
// Lists of <= 256 ids are rank-sorted in registers by one warp (up to eight ids per lane); longer ones by
// the whole CTA with a bitonic network in shared memory.
constexpr int SORT_WARPS = 8;
constexpr int SORT_PER_LANE = 8;
constexpr int SORT_WARP_MAX = 32 * SORT_PER_LANE;     // lists up to this length: one warp each, in registers
constexpr int WARP_SORT_SMEM = 1024;                  // ... up to this length: one warp each, in shared memory
__global__ void __launch_bounds__(SORT_WARPS * 32)
k_sort_tiles(const int32_t *__restrict__ tile_list, int cap, int32_t *__restrict__ pairs,
             const BinHeader *__restrict__ hdr) {
    pdl_trigger();      // (nr_kernels.h) the raster kernel behind this one
    __shared__ int s_ids[SMEM_SORT_CAP];
    __shared__ int s_long[SORT_WARPS * 32];
    __shared__ int s_nlong;
    if (hdr->overflow) return;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const TileList tl = open_tile_list(tile_list, cap);
    const int count = tl.total;

    // ---- pass A: lists of up to 256 ids, one warp per list, rank sort with the ids in registers
    // (warp_rank_sort reads the whole list before it writes, so sorting in place is safe)
    for (int w = blockIdx.x * SORT_WARPS + wid; w < count; w += gridDim.x * SORT_WARPS) {
        const int4 e = tile_entry(tl, w);
        const int n = e.w;
        if (n < 2 || n > SORT_WARP_MAX) continue;
        int32_t *a = pairs + e.z;
        if (n <= 32) warp_rank_sort<1>(a, n, a, lane);
        else if (n <= 64) warp_rank_sort<2>(a, n, a, lane);
        else if (n <= 128) warp_rank_sort<4>(a, n, a, lane);
        else warp_rank_sort<8>(a, n, a, lane);
    }

    // ---- pass A2: lists of 257 .. 1024 ids, still one warp per list (eight lists per CTA at a time, no
    // CTA barrier): bitonic network in the warp's 1024-id slice of shared memory, same direction over the
    // virtual power-of-two length (indices >= n behave as +inf and never move)
    // Only when there are more long lists than warps in the grid (a dense mesh everywhere): with a few
    // long lists (the limb of a sphere) one warp each would be the critical path, and pass B is faster.
    static_assert(SMEM_SORT_CAP >= SORT_WARPS * WARP_SORT_SMEM, "one slice per warp");
    const bool many_long = tl.c[0] > (int)gridDim.x * SORT_WARPS;
    const int warp_sort_max = many_long ? WARP_SORT_SMEM : SORT_WARP_MAX;
    for (int w = blockIdx.x * SORT_WARPS + wid; many_long && w < count; w += gridDim.x * SORT_WARPS) {
        const int4 e = tile_entry(tl, w);
        const int n = e.w;
        if (n <= SORT_WARP_MAX || n > WARP_SORT_SMEM) continue;
        int32_t *a = pairs + e.z;
        int *s = s_ids + wid * WARP_SORT_SMEM;
        for (int i = lane; i < n; i += 32) s[i] = a[i];
        __syncwarp();
        int lg = 9;
        while ((1 << lg) < n) ++lg;
        const int half = 1 << (lg - 1);
        for (int kk = 1; kk <= lg; ++kk) {
            const int k = 1 << kk;
            for (int i = lane; i < half; i += 32) {
                const int blk = i >> (kk - 1), off = i & ((k >> 1) - 1);
                const int lo = (blk << kk) + off, hi = (blk << kk) + k - 1 - off;
                if (hi < n) {
                    const int x = s[lo], y = s[hi];
                    if (x > y) { s[lo] = y; s[hi] = x; }
                }
            }
            __syncwarp();
            for (int jj = kk - 2; jj >= 0; --jj) {
                const int j = 1 << jj;
                for (int i = lane; i < half; i += 32) {
                    const int lo = ((i >> jj) << (jj + 1)) + (i & (j - 1)), hi = lo + j;
                    if (hi < n) {
                        const int x = s[lo], y = s[hi];
                        if (x > y) { s[lo] = y; s[hi] = x; }
                    }
                }
                __syncwarp();
            }
        }
        for (int i = lane; i < n; i += 32) a[i] = s[i];
        __syncwarp();
    }
    __syncthreads();

    // ---- pass B: longer lists, the whole CTA per list.  First every thread looks at one entry
    // of this CTA's share (independent loads), the long ones are compacted, then sorted one by one
    // with a same-direction bitonic network over a virtual power-of-two length (indices >= n behave
    // as +inf and never move).
    // (entry w belongs to CTA w % gridDim.x, so neighbouring, similarly long lists spread over CTAs)
    for (int base = 0; base * (int)gridDim.x + (int)blockIdx.x < count; base += blockDim.x) {
        if (tid == 0) s_nlong = 0;
        __syncthreads();
        const int w = (base + tid) * (int)gridDim.x + (int)blockIdx.x;
        if (w < count) {
            const int n = tile_entry(tl, w).w;
            if (n > warp_sort_max && n <= SMEM_SORT_CAP) s_long[atomicAdd(&s_nlong, 1)] = w;
        }
        __syncthreads();
        const int nlong = s_nlong;
        for (int li = 0; li < nlong; ++li) {
            const int4 e = tile_entry(tl, s_long[li]);
            const int n = e.w;
            int32_t *a = pairs + e.z;
            int unsorted = 0;
            for (int i = tid; i < n; i += blockDim.x) s_ids[i] = a[i];
            __syncthreads();
            for (int i = tid; i + 1 < n; i += blockDim.x) unsorted |= (s_ids[i] > s_ids[i + 1]);
            if (__syncthreads_or(unsorted)) {
                int lg = 8;
                while ((1 << lg) < n) ++lg;
                const int half = 1 << (lg - 1);
                for (int kk = 1; kk <= lg; ++kk) {
                    const int k = 1 << kk;
                    for (int i = tid; i < half; i += blockDim.x) {
                        const int blk = i >> (kk - 1), off = i & ((k >> 1) - 1);
                        const int lo = (blk << kk) + off, hi = (blk << kk) + k - 1 - off;
                        if (hi < n && s_ids[lo] > s_ids[hi]) {
                            const int t = s_ids[lo];
                            s_ids[lo] = s_ids[hi];
                            s_ids[hi] = t;
                        }
                    }
                    __syncthreads();
                    for (int jj = kk - 2; jj >= 0; --jj) {
                        const int j = 1 << jj;
                        for (int i = tid; i < half; i += blockDim.x) {
                            const int lo = ((i >> jj) << (jj + 1)) + (i & (j - 1)), hi = lo + j;
                            if (hi < n && s_ids[lo] > s_ids[hi]) {
                                const int t = s_ids[lo];
                                s_ids[lo] = s_ids[hi];
                                s_ids[hi] = t;
                            }
                        }
                        __syncthreads();
                    }
                }
                for (int i = tid; i < n; i += blockDim.x) a[i] = s_ids[i];
            }
            __syncthreads();
        }
        __syncthreads();
    }

    // ---- pass C (rare): lists longer than the shared-memory capacity, sorted in place in global
    // memory with the same network, one CTA per list
    if (hdr->max_tile_faces <= SMEM_SORT_CAP) return;
    for (int w = blockIdx.x; w < count; w += gridDim.x) {
        const int4 e = tile_entry(tl, w);
        const int n = e.w;
        if (n <= SMEM_SORT_CAP) continue;
        int32_t *a = pairs + e.z;
        int lg = 1;
        while ((1 << lg) < n) ++lg;
        const int half = 1 << (lg - 1);
        for (int kk = 1; kk <= lg; ++kk) {
            const int k = 1 << kk;
            for (int i = tid; i < half; i += blockDim.x) {
                const int blk = i >> (kk - 1), off = i & ((k >> 1) - 1);
                const int lo = (blk << kk) + off, hi = (blk << kk) + k - 1 - off;
                if (hi < n) {
                    const int x = a[lo], y = a[hi];
                    if (x > y) {
                        a[lo] = y;
                        a[hi] = x;
                    }
                }
            }
            __syncthreads();
            for (int jj = kk - 2; jj >= 0; --jj) {
                const int j = 1 << jj;
                for (int i = tid; i < half; i += blockDim.x) {
                    const int lo = ((i >> jj) << (jj + 1)) + (i & (j - 1)), hi = lo + j;
                    if (hi < n) {
                        const int x = a[lo], y = a[hi];
                        if (x > y) {
                            a[lo] = y;
                            a[hi] = x;
                        }
                    }
                }
                __syncthreads();
            }
        }
    }
}

bool binning_fits_one_cta_per_view(int nf, int R) {
    const int ntx = (R + TILE - 1) / TILE;
    return nf <= BINVIEW_MAX_FACES && ntx * ntx <= BINVIEW_MAX_TILES;
}

cudaError_t launch_binning(const BinningArgs &a, cudaStream_t stream) {
    const int nt = a.ntx * a.ntx;
    if (a.one_cta_per_view && a.tile_shift == 4 && binning_fits_one_cta_per_view(a.nf, a.R)) {
        static bool attr_set[64] = {false};
        const size_t smem = (4 * (size_t)nt + BINVIEW_SMEM_PAIRS) * sizeof(int);
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev >= 0 && dev < 64 && !attr_set[dev]) {
            cudaError_t e = cudaFuncSetAttribute(k_bin_view, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)((4 * (size_t)BINVIEW_MAX_TILES + BINVIEW_SMEM_PAIRS) * sizeof(int)));
            if (e != cudaSuccess) return e;
            attr_set[dev] = true;
        }
        cudaError_t e;
        {
            ProfScope p(PROF_MEMSET, stream);
            e = cudaMemsetAsync(a.hdr, 0, sizeof(BinHeader), stream);
            if (e == cudaSuccess) e = cudaMemsetAsync(a.tile_list, 0, sizeof(int32_t) * TILE_LIST_HDR, stream);
        }
        if (e != cudaSuccess) return e;
        // cluster size: as many CTAs per view as keep the whole grid in one wave (one CTA per SM), and no
        // more than the faces can use (a slice of fewer than 256 faces leaves most of a CTA idle)
        int cs = 1;
        while (cs < BINVIEW_MAX_CLUSTER && (long long)a.B * cs * 2 <= a.sm_count && a.nf > 256 * cs) cs *= 2;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(a.B * cs));
        cfg.blockDim = dim3(BINVIEW_THREADS);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)cs;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        {
            ProfScope p(PROF_SETUP, stream);
            e = cudaLaunchKernelEx(&cfg, k_bin_view, a.verts, a.faces, a.face_stride, a.nv, a.nf, a.R, a.draw_backside, a.ntx, a.rec,
                                   a.tile_count, a.pairs, a.pair_capacity, a.hdr, a.tile_list);
        }
        if (e == cudaSuccess) return e;
        // a device / partition that cannot co-schedule the cluster: nothing ran, take the general path
        (void)cudaGetLastError();
    }
    // header + tile counts are contiguous in the workspace: one memset
    cudaError_t e;
    {
        ProfScope p(PROF_MEMSET, stream);
        e = cudaMemsetAsync(a.hdr, 0, sizeof(BinHeader) + sizeof(int) * (size_t)a.B * nt, stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(a.tile_list, 0, sizeof(int32_t) * TILE_LIST_HDR, stream);
    }
    if (e != cudaSuccess) return e;
    const long long nface = (long long)a.B * a.nf;
    if (nface > 0) {
        const unsigned blocks = (unsigned)((nface + 255) / 256);
        ProfScope p(PROF_SETUP, stream);
        k_setup_count<<<blocks, 256, 0, stream>>>(a.verts, a.faces, a.face_stride, a.B, a.nv, a.nf, a.R,
                                                  a.draw_backside, a.rec, a.tile_count, a.ntx, a.tile_shift, a.hdr);
    }
    {
        ProfScope p(PROF_SCAN, stream);
        k_scan_tiles<<<a.B, 1024, 0, stream>>>(a.tile_count, a.tile_offset, a.tile_cursor, nt, a.ntx,
                                               a.pair_capacity, a.hdr, a.tile_list);
    }
    if (nface > 0) {
        const unsigned blocks = (unsigned)((nface + 255) / 256);
        {
            ProfScope p(PROF_SCATTER, stream);
            k_scatter<<<blocks, 256, 0, stream>>>(a.rec, a.B, a.nf, a.ntx, a.tile_shift, a.tile_cursor, a.pairs,
                                                  a.pair_capacity, a.hdr);
        }
        ProfScope p(PROF_SORT_LONG, stream);
        k_sort_tiles<<<a.sm_count * 8, SORT_WARPS * 32, 0, stream>>>(a.tile_list, a.B * nt, a.pairs, a.hdr);

    }
    return cudaGetLastError();
}

}  // namespace nr
