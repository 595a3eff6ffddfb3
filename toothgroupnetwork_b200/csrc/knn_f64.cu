// knn_f64.cu -- exact float64 k nearest neighbours (k <= 64) with scikit-learn KDTree semantics, plus a fused label vote.
//
// The tgnet inference pipeline asks a host KDTree for the k = 40 nearest of 24 000 sampled points for every raw-mesh
// vertex (10^5 - 2*10^5 queries) and counts how many of them carry the nearest one's label (the boundary step,
// inference_pipeline_tgn.py:289-330), then runs k = 1 label transfers (:107-140).  This file answers those queries on the
// device with the tree's arithmetic:
//
//      rdist = (dx*dx + dy*dy) + dz*dz   in float64, each operation rounded on its own (no FMA contraction)
//
// -- scikit-learn's EuclideanDistance.rdist and crop_knn.cu's dist_key -- ordered ascending by (rdist, index), so exact
// ties come out lower index first.  The k smallest under a total order do not depend on the order the candidates are met
// in, so the answer is the brute-force one whatever the traversal.
//
// Structure: the uniform grid of knn_grid.cu, built over a float32 copy of the points (tgn_knn_grid_build unchanged),
// followed by one pass that lays the float64 coordinates and row ids out in the grid's cell order.  One warp per query
// visits growing cubes of cells around it, keeping the k best in a sorted register list spread over the lanes
// (ceil(k/32) entries per lane), and stops once the k-th best rdist is provably below every unvisited point's.
//
// Cover bound.  Cells were assigned from float32 coordinates with float32 arithmetic, c = floor((x32 - ox) * inv_cs), so a
// point's true float64 x may lie slightly outside its cell [ox + c*cs, ox + (c+1)*cs).  With M the largest magnitude of
// the grid's box corners, |x - x32| <= 2^-24 M, the subtraction rounds by <= 2^-24 * 2M, and the product (inv_cs itself
// within 2^-24 of 1/cs) by <= 2 * 2^-24 * 2M in distance units: a point is within s0 = 7 * 2^-24 * M (< 4.2e-7 M) of its
// cell.  The kernel uses s = 4e-6 * (M + cs), ten times that, which also covers the float64 rounding of the face
// positions.  After the cube of cells [x0, x1] x [y0, y1] x [z0, z1] has been visited, an unvisited point lies in a cell
// beyond one of its faces, so its distance to the query is at least  gap = min over the faces that still have cells
// beyond them of (distance from the query to that face) - s.  The search stops when  tau < gap^2 * (1 - 1e-12)  with tau
// the k-th best rdist; the factor absorbs the rounding of rdist and of gap^2 (a few float64 ulps), and the strict
// comparison means no unvisited point can even tie with the k-th best.  A cube with no cells beyond any face is the
// whole grid.  The bound uses the query's own float64 position, so queries outside the points' bounding box (or far
// away from it) need no special case: the cube just grows until it covers them.
//
// Label vote (optional): with labels (n) float64, each query also writes nearest_label = labels[idx[0]] and
// is_boundary = (double)count / (double)k < ratio, count = how many of its k neighbours carry nearest_label, and counts
// the boundary queries in a device counter.  That is `count_unique_by_row(labels[idx])[:, 0] / k < ratio`
// (gen_utils.py:26-32: column 0 is the first occurrence of its own value, so it holds that value's count).
#include <cfloat>
#include <climits>

#include "common.cuh"
#include "knn_grid.cuh"
#include "tgn_b200.h"

namespace tgn {
namespace {

using knn_grid::GridWs;
using knn_grid::SegGrid;

constexpr int kWarps = 8;
constexpr int kMaxK = 64;
constexpr unsigned FULL = 0xffffffffu;

struct alignas(32) Rec {                   // one point in the grid's cell order
    double x, y, z;
    long long id;                          // original row
};

struct F64Ws {
    GridWs grid;
    float* xyz32;                          // [n][3]  float32 copy the grid is built from
    int* offset;                           // [1] = n
    Rec* rec;                              // [n]
};

size_t carve_f64(int n, F64Ws* ws, unsigned char* base)
{
    size_t off = knn_grid::carve(1, n, ws ? &ws->grid : nullptr, base);
    auto take = [&](size_t bytes) { const size_t o = off; off = (off + bytes + 255) & ~static_cast<size_t>(255); return o; };
    const size_t o_xyz = take(static_cast<size_t>(n) * 3 * sizeof(float));
    const size_t o_off = take(sizeof(int));
    const size_t o_rec = take(static_cast<size_t>(n) * sizeof(Rec));
    if (ws) {
        ws->xyz32 = reinterpret_cast<float*>(base + o_xyz);
        ws->offset = reinterpret_cast<int*>(base + o_off);
        ws->rec = reinterpret_cast<Rec*>(base + o_rec);
    }
    return off;
}

__global__ void __launch_bounds__(256) knn_f64_prep_kernel(int n, const double* __restrict__ pts, float* __restrict__ xyz32,
                                                           int* __restrict__ offset)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i == 0) offset[0] = n;
    if (i >= 3 * n) return;
    xyz32[i] = static_cast<float>(pts[i]);
}

__global__ void __launch_bounds__(256) knn_f64_records_kernel(int n, const double* __restrict__ pts, const float4* __restrict__ sorted,
                                                              Rec* __restrict__ rec)
{
    const int pos = blockIdx.x * 256 + threadIdx.x;
    if (pos >= n) return;
    const int id = __float_as_int(sorted[pos].w);
    Rec r;
    r.x = pts[3 * static_cast<size_t>(id)]; r.y = pts[3 * static_cast<size_t>(id) + 1]; r.z = pts[3 * static_cast<size_t>(id) + 2];
    r.id = id;
    rec[pos] = r;
}

__device__ __forceinline__ double rdist(double qx, double qy, double qz, const Rec& p) {
    const double dx = __dsub_rn(p.x, qx), dy = __dsub_rn(p.y, qy), dz = __dsub_rn(p.z, qz);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// (d, i) < (td, ti) in the (rdist, index) order
__device__ __forceinline__ bool before(double d, int i, double td, int ti) { return d < td || (d == td && i < ti); }

__device__ __forceinline__ int cell_index(double v, float o, float inv_cs) {
    const double c = floor((v - static_cast<double>(o)) * static_cast<double>(inv_cs));
    return static_cast<int>(fmin(fmax(c, -16777216.0), 16777216.0));      // far-away queries: keep the cube arithmetic in int
}

template <int EPL>
__global__ void __launch_bounds__(kWarps * 32)
knn_f64_query_kernel(int m, int k, const double* __restrict__ queries, const Rec* __restrict__ rec, const int* __restrict__ cst,
                     const SegGrid* __restrict__ segp, int64_t* __restrict__ idx, double* __restrict__ dist,
                     const double* __restrict__ labels, double ratio, double* __restrict__ nearest_label,
                     unsigned char* __restrict__ is_boundary, int* __restrict__ n_boundary)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = blockIdx.x * kWarps + warp;
    if (q >= m) return;                                   // warps are independent: no block-level barriers below
    const double qx = queries[3 * static_cast<size_t>(q)], qy = queries[3 * static_cast<size_t>(q) + 1],
                 qz = queries[3 * static_cast<size_t>(q) + 2];
    const SegGrid g = *segp;

    // entry lane*EPL + e of the ascending list; entries >= k only ever hold what was pushed out of the first k
    double ld[EPL];
    int li[EPL];
#pragma unroll
    for (int e = 0; e < EPL; ++e) { ld[e] = DBL_MAX; li[e] = INT_MAX; }
    const int kth_lane = (k - 1) / EPL, kth_sub = (k - 1) % EPL;
    double tau = DBL_MAX;                                 // the k-th best so far
    int tau_i = INT_MAX;

    // slack of the cover bound (header comment)
    const float mx = fmaxf(fabsf(g.ox), fabsf(g.ox + g.nx * g.cs)), my = fmaxf(fabsf(g.oy), fabsf(g.oy + g.ny * g.cs)),
                mz = fmaxf(fabsf(g.oz), fabsf(g.oz + g.nz * g.cs));
    const double slack = 4e-6 * (static_cast<double>(fmaxf(mx, fmaxf(my, mz))) + static_cast<double>(g.cs));
    const double cs = g.cs;

    const int cx = cell_index(qx, g.ox, g.inv_cs), cy = cell_index(qy, g.oy, g.inv_cs), cz = cell_index(qz, g.oz, g.inv_cs);
    int R0 = 1;                                           // first cube that reaches the grid at all
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
                // the row's unvisited candidates: the whole x range, or only the cells beyond the previous cube's x range
                int ranges[2][2] = {{0, 0}, {0, 0}};
                if (!old_row) {
                    if (x0 <= x1) { ranges[0][0] = __ldg(cst + row + x0); ranges[0][1] = __ldg(cst + row + x1 + 1); }
                } else {
                    const int xl1 = min(cx - Rprev - 1, g.nx - 1), xr0 = max(cx + Rprev + 1, 0);
                    if (x0 <= xl1) { ranges[0][0] = __ldg(cst + row + x0); ranges[0][1] = __ldg(cst + row + xl1 + 1); }
                    if (xr0 <= x1) { ranges[1][0] = __ldg(cst + row + xr0); ranges[1][1] = __ldg(cst + row + x1 + 1); }
                }
#pragma unroll 1
                for (int part = 0; part < 2; ++part) {
                    const int p0 = part ? ranges[1][0] : ranges[0][0], p1 = part ? ranges[1][1] : ranges[0][1];
                    for (int o = p0; o < p1; o += 32) {
                        const int i = o + lane;
                        double d = DBL_MAX;
                        int ci_lane = INT_MAX;
                        if (i < p1) {
                            const Rec r = rec[i];
                            d = rdist(qx, qy, qz, r);
                            ci_lane = static_cast<int>(r.id);
                        }
                        unsigned mask = __ballot_sync(FULL, i < p1 && before(d, ci_lane, tau, tau_i));
                        while (mask) {
                            const int src = __ffs(mask) - 1;
                            mask &= mask - 1;
                            const double cd = __shfl_sync(FULL, d, src);
                            const int ci = __shfl_sync(FULL, ci_lane, src);
                            if (!before(cd, ci, tau, tau_i)) continue;
                            int below = 0;
#pragma unroll
                            for (int e = 0; e < EPL; ++e) below += before(ld[e], li[e], cd, ci) ? 1 : 0;
                            const int plane = __popc(__ballot_sync(FULL, below == EPL));
                            const double up_d = __shfl_up_sync(FULL, ld[EPL - 1], 1);
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
                            double td = ld[0];
                            int ti = li[0];
#pragma unroll
                            for (int e = 1; e < EPL; ++e) if (kth_sub == e) { td = ld[e]; ti = li[e]; }
                            tau = __shfl_sync(FULL, td, kth_lane);
                            tau_i = __shfl_sync(FULL, ti, kth_lane);
                        }
                    }
                }
            }
        }
        Rprev = R;
        double gap = DBL_MAX;
        if (x0 > 0) gap = fmin(gap, qx - (static_cast<double>(g.ox) + x0 * cs));
        if (x1 < g.nx - 1) gap = fmin(gap, (static_cast<double>(g.ox) + (x1 + 1) * cs) - qx);
        if (y0 > 0) gap = fmin(gap, qy - (static_cast<double>(g.oy) + y0 * cs));
        if (y1 < g.ny - 1) gap = fmin(gap, (static_cast<double>(g.oy) + (y1 + 1) * cs) - qy);
        if (z0 > 0) gap = fmin(gap, qz - (static_cast<double>(g.oz) + z0 * cs));
        if (z1 < g.nz - 1) gap = fmin(gap, (static_cast<double>(g.oz) + (z1 + 1) * cs) - qz);
        if (gap == DBL_MAX) break;                        // whole grid visited
        gap -= slack;
        if (gap > 0.0 && tau < gap * gap * (1.0 - 1e-12)) break;
    }

    if (idx || dist) {
#pragma unroll
        for (int e = 0; e < EPL; ++e) {
            const int ent = lane * EPL + e;
            if (ent < k) {
                if (idx) idx[static_cast<size_t>(q) * k + ent] = li[e];
                if (dist) dist[static_cast<size_t>(q) * k + ent] = __dsqrt_rn(ld[e]);
            }
        }
    }
    if (labels) {
        const int i0 = __shfl_sync(FULL, li[0], 0);
        const double nl = __ldg(labels + i0);
        int cnt = 0;
#pragma unroll
        for (int e = 0; e < EPL; ++e) {
            const int ent = lane * EPL + e;
            if (ent < k && __ldg(labels + li[e]) == nl) ++cnt;
        }
        cnt = __reduce_add_sync(FULL, cnt);
        if (lane == 0) {
            const bool bd = __ddiv_rn(static_cast<double>(cnt), static_cast<double>(k)) < ratio;
            nearest_label[q] = nl;
            is_boundary[q] = bd ? 1 : 0;
            if (bd) atomicAdd(n_boundary, 1);
        }
    }
}

}  // namespace
}  // namespace tgn

extern "C" {

size_t tgn_knn_f64_bytes(int n)
{
    return tgn::carve_f64(n, nullptr, nullptr);
}

int tgn_knn_f64_build(int n, const double* points, void* workspace, void* stream)
{
    using namespace tgn;
    if (n <= 0) return TGN_OK;
    if (!points || !workspace) { set_error("knn_f64_build: null argument"); return TGN_ERR_INVALID; }
    if (n > INT_MAX / 3) { set_error("knn_f64_build: n=%d too large", n); return TGN_ERR_INVALID; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    F64Ws ws{};
    carve_f64(n, &ws, static_cast<unsigned char*>(workspace));
    knn_f64_prep_kernel<<<(3 * n + 255) / 256, 256, 0, st>>>(n, points, ws.xyz32, ws.offset);
    int rc = check_launch("knn_f64_prep_kernel");
    if (rc != TGN_OK) return rc;
    if ((rc = tgn_knn_grid_build(1, n, ws.xyz32, ws.offset, workspace, stream)) != TGN_OK) return rc;
    knn_f64_records_kernel<<<(n + 255) / 256, 256, 0, st>>>(n, points, ws.grid.sorted, ws.rec);
    return check_launch("knn_f64_records_kernel");
}

int tgn_knn_f64_query(int n, int m, int k, const double* queries, const void* workspace, int64_t* idx, double* dist,
                      const double* labels, double ratio, double* nearest_label, unsigned char* is_boundary, int* n_boundary,
                      void* stream)
{
    using namespace tgn;
    if (k <= 0 || k > kMaxK) { set_error("knn_f64_query: k=%d outside [1, %d]", k, kMaxK); return TGN_ERR_INVALID; }
    if (k > n) { set_error("knn_f64_query: k=%d exceeds the %d points", k, n); return TGN_ERR_INVALID; }
    if (!workspace || (m > 0 && !queries)) { set_error("knn_f64_query: null argument"); return TGN_ERR_INVALID; }
    if (labels && (!nearest_label || !is_boundary || !n_boundary)) {
        set_error("knn_f64_query: labels given without nearest_label / is_boundary / n_boundary");
        return TGN_ERR_INVALID;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (labels && cudaMemsetAsync(n_boundary, 0, sizeof(int), st) != cudaSuccess) {
        set_error("knn_f64_query: cudaMemsetAsync failed");
        return TGN_ERR_CUDA;
    }
    if (m <= 0) return TGN_OK;
    F64Ws ws{};
    carve_f64(n, &ws, const_cast<unsigned char*>(static_cast<const unsigned char*>(workspace)));
    const int grid = (m + kWarps - 1) / kWarps;
    if (k <= 32)
        knn_f64_query_kernel<1><<<grid, kWarps * 32, 0, st>>>(m, k, queries, ws.rec, ws.grid.cell_start, ws.grid.seg, idx, dist,
                                                             labels, ratio, nearest_label, is_boundary, n_boundary);
    else
        knn_f64_query_kernel<2><<<grid, kWarps * 32, 0, st>>>(m, k, queries, ws.rec, ws.grid.cell_start, ws.grid.seg, idx, dist,
                                                             labels, ratio, nearest_label, is_boundary, n_boundary);
    return check_launch("knn_f64_query_kernel");
}

}  // extern "C"
