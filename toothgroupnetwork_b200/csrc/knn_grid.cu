// knn_grid.cu -- k nearest neighbours through a per-segment uniform grid (exact, same answers as knn.cu).
//
// knn.cu scans the whole segment for every query: 5.8e8 distance evaluations for the 24 000 x 24 000, k = 36
// search tgnet_fps issues five times per forward (blocks.py:34-35).  A query's k nearest lie within a few cells of
// it, so this file bins every segment's points into a uniform grid once (counting sort, cell-sorted float4 records
// carrying the original row id) and lets a warp visit growing cubes of cells around its query until the (k+1)-th
// best distance found so far is provably covered:
//
//      after the cube of radius R cells around the query's cell has been visited, every unvisited point is at
//      least R * cell_size away, so the search stops once  d2[(k+1)-th best] <= (R * cell_size)^2 * (1 - 1e-5)
//
// (the slack covers the rounding of the comparison; stopping later only costs time).  Candidates are tested with the
// reference's arithmetic (FMUL dy*dy, FFMA dx*dx+., FFMA dz*dz+., knnquery_cuda_kernel.cu:84-87 as compiled) and
// kept in the same register-resident sorted list as knn.cu.  With distinct distances the k smallest in ascending order
// do not depend on the visiting order, so the result IS the reference's; if two of the k+1 best tie, the reference's
// answer depends on its heap history (index-order scan, :21-48) and the warp re-runs that query with the exact heap
// emulation over the whole segment, exactly as knn.cu does.  Segments shorter than k end up visiting everything and
// keep (segment start, 1e10) in the trailing slots (:88-91).
//
// The grid depends only on (xyz, offset): the Python layer builds it once per point set and reuses it for every kNN
// against that set (self k=36 and k=24 searches, the strided TransitionDown queries, k=3 / k=1 up-sampling).
#include <algorithm>
#include <climits>

#include "common.cuh"
#include "knn_grid.cuh"
#include "tgn_b200.h"

namespace tgn {
namespace {

using knn_grid::carve;
using knn_grid::GridWs;
using knn_grid::kCellsMax;
using knn_grid::SegGrid;

constexpr int kWarps = 8;
constexpr int kMaxK = 128;
constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ int float_ordered(float f) {
    const int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float ordered_float(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

__device__ __forceinline__ int cell_coord(float v, float org, float inv_cs, int n) {
    const int c = static_cast<int>(floorf((v - org) * inv_cs));
    return min(max(c, 0), n - 1);
}

// ---- 1. bounding box, cell size, zeroed counters: one CTA per segment --------------------------------------------
__global__ void __launch_bounds__(256) knn_grid_setup_kernel(const float* __restrict__ xyz, const int* __restrict__ offset, GridWs ws)
{
    __shared__ int red[6][8];
    __shared__ int s_cells;
    const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int start = s ? offset[s - 1] : 0, end = offset[s];
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = start + tid; i < end; i += 256) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float v = __ldg(xyz + 3 * static_cast<size_t>(i) + a);
            mn[a] = fminf(mn[a], v); mx[a] = fmaxf(mx[a], v);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const int lo = __reduce_min_sync(FULL, float_ordered(mn[a])), hi = __reduce_max_sync(FULL, float_ordered(mx[a]));
        if (lane == 0) { red[a][warp] = lo; red[3 + a][warp] = hi; }
    }
    __syncthreads();
    if (tid == 0) {
        float lo[3], ext[3], emax = 0.f;
        for (int a = 0; a < 3; ++a) {
            int l = red[a][0], h = red[3 + a][0];
            for (int w = 1; w < 8; ++w) { l = min(l, red[a][w]); h = max(h, red[3 + a][w]); }
            lo[a] = ordered_float(l);
            ext[a] = ordered_float(h) - lo[a];
            emax = fmaxf(emax, ext[a]);
        }
        const int n = end - start;
        SegGrid g;
        g.ox = lo[0]; g.oy = lo[1]; g.oz = lo[2];
        g.nx = g.ny = g.nz = 1;
        g.cs = 1.f;
        if (n > 0 && emax > 0.f && isfinite(emax)) {
            // about two points per cell of the bounding box (a surface-like cloud fills a fraction of them, which
            // leaves ~10-20 points in the occupied ones), never more than kCellsMax cells
            const float target = fminf(fmaxf(0.5f * n, 1.f), static_cast<float>(kCellsMax));
            float vol = 1.f;
            for (int a = 0; a < 3; ++a) vol *= fmaxf(ext[a], 1e-3f * emax);
            float cs = cbrtf(vol / target);
            for (int it = 0; it < 200; ++it) {
                const float fx = ext[0] / cs, fy = ext[1] / cs, fz = ext[2] / cs;
                if (fx < 2048.f && fy < 2048.f && fz < 2048.f) {
                    g.nx = static_cast<int>(fx) + 1; g.ny = static_cast<int>(fy) + 1; g.nz = static_cast<int>(fz) + 1;
                    if (static_cast<long long>(g.nx) * g.ny * g.nz <= kCellsMax) break;
                }
                g.nx = g.ny = g.nz = 1;
                cs *= 1.26f;
            }
            g.cs = cs;
        }
        g.inv_cs = 1.0f / g.cs;
        ws.seg[s] = g;
        s_cells = g.nx * g.ny * g.nz;
    }
    __syncthreads();
    int* cur = ws.cursor + static_cast<size_t>(s) * kCellsMax;
    for (int c = tid; c < s_cells; c += 256) cur[c] = 0;
}

__device__ __forceinline__ int segment_of(int i, const int* __restrict__ offset, int b) {
    int s = 0;
    while (s < b - 1 && i >= __ldg(offset + s)) ++s;
    return s;
}

// ---- 2. histogram ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) knn_grid_count_kernel(int n_total, int b, const float* __restrict__ xyz,
                                                             const int* __restrict__ offset, GridWs ws)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n_total) return;
    const int s = segment_of(i, offset, b);
    const SegGrid g = ws.seg[s];
    const float x = __ldg(xyz + 3 * static_cast<size_t>(i)), y = __ldg(xyz + 3 * static_cast<size_t>(i) + 1), z = __ldg(xyz + 3 * static_cast<size_t>(i) + 2);
    const int c = (cell_coord(z, g.oz, g.inv_cs, g.nz) * g.ny + cell_coord(y, g.oy, g.inv_cs, g.ny)) * g.nx + cell_coord(x, g.ox, g.inv_cs, g.nx);
    ws.cell_of[i] = c;
    atomicAdd(ws.cursor + static_cast<size_t>(s) * kCellsMax + c, 1);
}

// ---- 3. exclusive scan of a segment's counters: one CTA (1024 threads) per segment -------------------------------------
__global__ void __launch_bounds__(1024) knn_grid_scan_kernel(const int* __restrict__ offset, GridWs ws)
{
    __shared__ int warp_tot[32];
    const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const SegGrid g = ws.seg[s];
    const int cells = g.nx * g.ny * g.nz;
    const int start = s ? offset[s - 1] : 0;
    int* cur = ws.cursor + static_cast<size_t>(s) * kCellsMax;
    int* cst = ws.cell_start + static_cast<size_t>(s) * (kCellsMax + 1);
    constexpr int kPer = kCellsMax / 1024;           // 32 consecutive cells per thread
    int v[kPer], sum = 0;
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
        const int c = tid * kPer + i;
        v[i] = c < cells ? cur[c] : 0;
        sum += v[i];
    }
    int incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = warp_tot[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(FULL, w, d);
            if (lane >= d) w += t;
        }
        warp_tot[lane] = w;
    }
    __syncthreads();
    int run = start + (incl - sum) + (warp ? warp_tot[warp - 1] : 0);
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
        const int c = tid * kPer + i;
        if (c < cells) { cst[c] = run; cur[c] = run; }
        run += v[i];
    }
    if (tid == 1023) cst[cells] = run;               // == segment end
}

// ---- 4. scatter ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) knn_grid_scatter_kernel(int n_total, int b, const float* __restrict__ xyz,
                                                               const int* __restrict__ offset, GridWs ws)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n_total) return;
    const int s = segment_of(i, offset, b);
    const int pos = atomicAdd(ws.cursor + static_cast<size_t>(s) * kCellsMax + ws.cell_of[i], 1);
    ws.sorted[pos] = make_float4(__ldg(xyz + 3 * static_cast<size_t>(i)), __ldg(xyz + 3 * static_cast<size_t>(i) + 1),
                                 __ldg(xyz + 3 * static_cast<size_t>(i) + 2), __int_as_float(i));
}

// ---- 5. query ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float sq_dist_direct(float qx, float qy, float qz, float x, float y, float z) {
    const float dx = qx - x, dy = qy - y, dz = qz - z;
    float d = __fmul_rn(dy, dy);
    d = __fmaf_rn(dx, dx, d);
    return __fmaf_rn(dz, dz, d);
}
__device__ __forceinline__ void heap_sift_down(float* d, int* id, int len) {      // as in knn.cu / the reference's reheap
    int parent = 0;
    for (;;) {
        int kid = 2 * parent + 1;
        if (kid >= len) return;
        if (kid + 1 < len && d[kid + 1] > d[kid]) ++kid;
        if (d[parent] > d[kid]) return;
        const float fd = d[parent]; d[parent] = d[kid]; d[kid] = fd;
        const int fi = id[parent]; id[parent] = id[kid]; id[kid] = fi;
        parent = kid;
    }
}

template <int EPL>
__global__ void __launch_bounds__(kWarps * 32)
knn_grid_query_kernel(int b, int m, int k, const float* __restrict__ xyz, const float* __restrict__ new_xyz,
                      const int* __restrict__ offset, const int* __restrict__ new_offset, const GridWs ws,
                      int* __restrict__ idx, float* __restrict__ dist2)
{
    __shared__ float hd[kWarps][kMaxK];
    __shared__ int hi[kWarps][kMaxK];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = blockIdx.x * kWarps + warp;
    if (q >= m) return;                                   // warps are independent: no block-level barriers below
    const int seg = segment_of(q, new_offset, b);
    const int start = seg ? __ldg(offset + seg - 1) : 0, end = __ldg(offset + seg);
    const float qx = __ldg(new_xyz + 3 * static_cast<size_t>(q)), qy = __ldg(new_xyz + 3 * static_cast<size_t>(q) + 1),
                qz = __ldg(new_xyz + 3 * static_cast<size_t>(q) + 2);
    const SegGrid g = ws.seg[seg];
    const int* __restrict__ cst = ws.cell_start + static_cast<size_t>(seg) * (kCellsMax + 1);

    float ld[EPL];
    int li[EPL];
#pragma unroll
    for (int i = 0; i < EPL; ++i) { ld[i] = 1e10f; li[i] = start; }
    const int kth_lane = k / EPL, kth_sub = k % EPL;
    float tau = 1e10f;

    auto scan_range = [&](int p0, int p1) {               // candidates sorted[p0, p1)
        for (int o = p0; o < p1; o += 32) {
            const int i = o + lane;
            float d = 1e30f;
            int ci_lane = 0;
            if (i < p1) {
                const float4 c = __ldg(ws.sorted + i);
                d = sq_dist_direct(qx, qy, qz, c.x, c.y, c.z);
                ci_lane = __float_as_int(c.w);
            }
            unsigned mask = __ballot_sync(FULL, d < tau);
            while (mask) {
                const int src = __ffs(mask) - 1;
                mask &= mask - 1;
                const float cd = __shfl_sync(FULL, d, src);
                const int ci = __shfl_sync(FULL, ci_lane, src);
                if (cd < tau) {
                    int below = 0;
#pragma unroll
                    for (int e = 0; e < EPL; ++e) below += (ld[e] <= cd) ? 1 : 0;
                    const unsigned full_lanes = __ballot_sync(FULL, below == EPL);
                    const int plane = __popc(full_lanes);
                    const float up_d = __shfl_up_sync(FULL, ld[EPL - 1], 1);
                    const int up_i = __shfl_up_sync(FULL, li[EPL - 1], 1);
                    if (lane > plane) {
#pragma unroll
                        for (int e = EPL - 1; e > 0; --e) { ld[e] = ld[e - 1]; li[e] = li[e - 1]; }
                        ld[0] = up_d; li[0] = up_i;
                    } else if (lane == plane) {
#pragma unroll
                        for (int e = EPL - 1; e > 0; --e) {
                            if (e > below) { ld[e] = ld[e - 1]; li[e] = li[e - 1]; }
                        }
#pragma unroll
                        for (int e = 0; e < EPL; ++e)
                            if (e == below) { ld[e] = cd; li[e] = ci; }
                    }
                    float tl = ld[0];
#pragma unroll
                    for (int e = 1; e < EPL; ++e) tl = (kth_sub == e) ? ld[e] : tl;
                    tau = __shfl_sync(FULL, tl, kth_lane);
                }
            }
        }
    };

    // the query's (unclamped) cell; cubes of growing radius around it
    const int cx = static_cast<int>(floorf((qx - g.ox) * g.inv_cs)), cy = static_cast<int>(floorf((qy - g.oy) * g.inv_cs)),
              cz = static_cast<int>(floorf((qz - g.oz) * g.inv_cs));
    // first radius worth visiting: the cube must reach the grid at all
    int R0 = 1;
    R0 = max(R0, max(-cx, cx - (g.nx - 1)));
    R0 = max(R0, max(-cy, cy - (g.ny - 1)));
    R0 = max(R0, max(-cz, cz - (g.nz - 1)));
    int Rprev = -1;                                       // nothing visited yet
    for (int R = R0;; ++R) {
        const int z0 = max(cz - R, 0), z1 = min(cz + R, g.nz - 1), y0 = max(cy - R, 0), y1 = min(cy + R, g.ny - 1);
        const int x0 = max(cx - R, 0), x1 = min(cx + R, g.nx - 1);
        for (int z = z0; z <= z1; ++z) {
            const bool z_old = Rprev >= 0 && z >= cz - Rprev && z <= cz + Rprev;
            for (int y = y0; y <= y1; ++y) {
                const int row = (z * g.ny + y) * g.nx;
                const bool old_row = z_old && y >= cy - Rprev && y <= cy + Rprev;
                if (!old_row) {
                    if (x0 <= x1) scan_range(__ldg(cst + row + x0), __ldg(cst + row + x1 + 1));
                } else {                                   // only the cells beyond the previous cube's x range are new
                    const int xl1 = min(cx - Rprev - 1, g.nx - 1), xr0 = max(cx + Rprev + 1, 0);
                    if (x0 <= xl1) scan_range(__ldg(cst + row + x0), __ldg(cst + row + xl1 + 1));
                    if (xr0 <= x1) scan_range(__ldg(cst + row + xr0), __ldg(cst + row + x1 + 1));
                }
            }
        }
        Rprev = R;
        const float cover = static_cast<float>(R) * g.cs;
        if (tau <= cover * cover * 0.99999f) break;                       // the (k+1)-th best is covered
        if (cx - R <= 0 && cy - R <= 0 && cz - R <= 0 && cx + R >= g.nx - 1 && cy + R >= g.ny - 1 && cz + R >= g.nz - 1) break;   // whole grid visited
    }

    // ---- tie check / output / exact heap emulation: identical to knn.cu ---------------------------------------------
    bool tie = false;
    {
        const float prev_last = __shfl_up_sync(FULL, ld[EPL - 1], 1);
#pragma unroll
        for (int e = 0; e < EPL; ++e) {
            const int ent = lane * EPL + e;
            const float prev = e ? ld[e - 1] : prev_last;
            if (ent >= 1 && ent <= k && ld[e] == prev && ld[e] < 1e10f) tie = true;
        }
        tie = __any_sync(FULL, tie);
    }
    int* orow = idx + static_cast<size_t>(q) * k;
    float* drow = dist2 + static_cast<size_t>(q) * k;
    if (!tie) {
#pragma unroll
        for (int e = 0; e < EPL; ++e) {
            const int ent = lane * EPL + e;
            if (ent < k) { orow[ent] = li[e]; drow[ent] = ld[e]; }
        }
        return;
    }
    float* d_heap = hd[warp];
    int* i_heap = hi[warp];
    for (int e = lane; e < k; e += 32) { d_heap[e] = 1e10f; i_heap[e] = start; }
    __syncwarp();
    for (int o = start; o < end; o += 32) {
        const int i = o + lane;
        float d = 1e30f;
        if (i < end) d = sq_dist_direct(qx, qy, qz, __ldg(xyz + 3 * static_cast<size_t>(i)), __ldg(xyz + 3 * static_cast<size_t>(i) + 1),
                                        __ldg(xyz + 3 * static_cast<size_t>(i) + 2));
        unsigned mask = __ballot_sync(FULL, d < d_heap[0]);
        while (mask) {
            const int src = __ffs(mask) - 1;
            mask &= mask - 1;
            const float cd = __shfl_sync(FULL, d, src);
            if (lane == 0 && cd < d_heap[0]) {
                d_heap[0] = cd; i_heap[0] = o + src;
                heap_sift_down(d_heap, i_heap, k);
            }
            __syncwarp();
        }
    }
    if (lane == 0) {
        for (int last = k - 1; last > 0; --last) {
            const float fd = d_heap[0]; d_heap[0] = d_heap[last]; d_heap[last] = fd;
            const int fi = i_heap[0]; i_heap[0] = i_heap[last]; i_heap[last] = fi;
            heap_sift_down(d_heap, i_heap, last);
        }
    }
    __syncwarp();
    for (int e = lane; e < k; e += 32) { orow[e] = i_heap[e]; drow[e] = d_heap[e]; }
}

}  // namespace
}  // namespace tgn

extern "C" {

size_t tgn_knn_grid_bytes(int b, int n_total)
{
    return tgn::carve(b, n_total, nullptr, nullptr);
}

int tgn_knn_grid_build(int b, int n_total, const float* xyz, const int* offset, void* workspace, void* stream)
{
    using namespace tgn;
    if (b <= 0 || n_total <= 0) return TGN_OK;
    if (!xyz || !offset || !workspace) { set_error("knn_grid_build: null argument"); return TGN_ERR_INVALID; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GridWs ws{};
    carve(b, n_total, &ws, static_cast<unsigned char*>(workspace));
    knn_grid_setup_kernel<<<b, 256, 0, st>>>(xyz, offset, ws);
    int rc = check_launch("knn_grid_setup_kernel");
    if (rc != TGN_OK) return rc;
    const int blocks = (n_total + 255) / 256;
    knn_grid_count_kernel<<<blocks, 256, 0, st>>>(n_total, b, xyz, offset, ws);
    if ((rc = check_launch("knn_grid_count_kernel")) != TGN_OK) return rc;
    knn_grid_scan_kernel<<<b, 1024, 0, st>>>(offset, ws);
    if ((rc = check_launch("knn_grid_scan_kernel")) != TGN_OK) return rc;
    knn_grid_scatter_kernel<<<blocks, 256, 0, st>>>(n_total, b, xyz, offset, ws);
    return check_launch("knn_grid_scatter_kernel");
}

int tgn_knn_grid_query(int b, int n_total, int m, int nsample, const float* xyz, const float* new_xyz, const int* offset,
                       const int* new_offset, const void* workspace, int* idx, float* dist2, void* stream)
{
    using namespace tgn;
    if (m <= 0 || nsample <= 0) return TGN_OK;
    if (nsample > kMaxK - 1) { set_error("knnquery: nsample=%d exceeds %d", nsample, kMaxK - 1); return TGN_ERR_INVALID; }
    if (b <= 0 || !workspace) { set_error("knn_grid_query: bad arguments"); return TGN_ERR_INVALID; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GridWs ws{};
    carve(b, n_total, &ws, const_cast<unsigned char*>(static_cast<const unsigned char*>(workspace)));
    const int grid = (m + kWarps - 1) / kWarps;
    const int epl = (nsample + 1 + 31) / 32;
    switch (epl) {
        case 1: knn_grid_query_kernel<1><<<grid, kWarps * 32, 0, st>>>(b, m, nsample, xyz, new_xyz, offset, new_offset, ws, idx, dist2); break;
        case 2: knn_grid_query_kernel<2><<<grid, kWarps * 32, 0, st>>>(b, m, nsample, xyz, new_xyz, offset, new_offset, ws, idx, dist2); break;
        case 3: knn_grid_query_kernel<3><<<grid, kWarps * 32, 0, st>>>(b, m, nsample, xyz, new_xyz, offset, new_offset, ws, idx, dist2); break;
        default: knn_grid_query_kernel<4><<<grid, kWarps * 32, 0, st>>>(b, m, nsample, xyz, new_xyz, offset, new_offset, ws, idx, dist2); break;
    }
    return check_launch("knn_grid_query_kernel");
}

}  // extern "C"
