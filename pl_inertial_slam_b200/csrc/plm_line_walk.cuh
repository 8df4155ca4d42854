// The Bresenham walk of StVO::GridStructure's line fill, shared by the grid builders on the device: the stereo-frame
// pipeline (plm_frames.cuh, shared-memory grid of the right image) and the keyframe grids of the resident local map
// (plm_localmap.cuh, grids in global memory).
#pragma once
#include "plm_common.cuh"

namespace plm {

// lineIterator.cpp:34-77 + gridStructure.cpp:33-41: Bresenham from double endpoints; first cell and
// last column come from truncation of the (possibly swapped) endpoints, error starts at dx / 2.
// The walk is cut after max_steps cells (the host rejects frames with longer walks).
template <class F>
__device__ __forceinline__ void line_walk(double x1, double y1, double x2, double y2, int max_steps, F &&f) {
    const bool steep = fabs(__dsub_rn(y2, y1)) > fabs(__dsub_rn(x2, x1));
    if (steep) {
        double t = x1; x1 = y1; y1 = t;
        t = x2; x2 = y2; y2 = t;
    }
    if (x1 > x2) {
        double t = x1; x1 = x2; x2 = t;
        t = y1; y1 = y2; y2 = t;
    }
    const double dx = __dsub_rn(x2, x1), dy = fabs(__dsub_rn(y2, y1));
    double error = __ddiv_rn(dx, 2.0);
    const int ystep = (y1 < y2) ? 1 : -1;
    int y = static_cast<int>(y1), x = static_cast<int>(x1);
    const int max_x = static_cast<int>(x2);
    for (int s = 0; x <= max_x && s < max_steps; ++x, ++s) {
        f(steep ? y : x, steep ? x : y);
        error = __dsub_rn(error, dy);
        if (error < 0) {
            y += ystep;
            error = __dadd_rn(error, dx);
        }
    }
}

} // namespace plm
