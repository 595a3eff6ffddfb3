// knn_grid.cuh -- layout of the uniform-grid workspace built by tgn_knn_grid_build (knn_grid.cu).
//
// Shared with knn_f64.cu, which builds the same grid over a float32 copy of its float64 points and then reads the cell
// ranges (cell_start) and the per-segment geometry (seg) back out of the workspace.
#pragma once

#include <cstddef>

namespace tgn {
namespace knn_grid {

constexpr int kCellsMax = 32768;          // cells per segment

struct SegGrid {
    float ox, oy, oz, inv_cs;
    float cs;
    int nx, ny, nz;
};

struct GridWs {                            // all arrays live in one caller-provided workspace
    float4* sorted;                        // [n_total]  (x, y, z, original row id as int bits), cell-sorted per segment
    int* cell_of;                          // [n_total]
    int* cell_start;                       // [b][kCellsMax + 1]  global positions into `sorted`
    int* cursor;                           // [b][kCellsMax]
    SegGrid* seg;                          // [b]
};

inline size_t carve(int b, int n_total, GridWs* ws, unsigned char* base)
{
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off = (off + bytes + 255) & ~static_cast<size_t>(255); return o; };
    const size_t o_sorted = take(static_cast<size_t>(n_total) * sizeof(float4));
    const size_t o_cell = take(static_cast<size_t>(n_total) * sizeof(int));
    const size_t o_start = take(static_cast<size_t>(b) * (kCellsMax + 1) * sizeof(int));
    const size_t o_cur = take(static_cast<size_t>(b) * kCellsMax * sizeof(int));
    const size_t o_seg = take(static_cast<size_t>(b) * sizeof(SegGrid));
    if (ws) {
        ws->sorted = reinterpret_cast<float4*>(base + o_sorted);
        ws->cell_of = reinterpret_cast<int*>(base + o_cell);
        ws->cell_start = reinterpret_cast<int*>(base + o_start);
        ws->cursor = reinterpret_cast<int*>(base + o_cur);
        ws->seg = reinterpret_cast<SegGrid*>(base + o_seg);
    }
    return off;
}

}  // namespace knn_grid
}  // namespace tgn
