// Host side of the frame grids the frame call returns (hvo_frame_grid_outputs): Frame::AssignFeaturesToGrid and
// Frame::AssignFeaturesToGridForLine (reference src/Frame.cc:832-872) fill
//
//     std::vector<std::size_t> mGrid[FRAME_GRID_COLS][FRAME_GRID_ROWS];          // 64 x 48
//     std::vector<std::size_t> mGridForLine[FRAME_GRID_COLS][FRAME_GRID_ROWS];
//
// with each cell's feature indices in push_back (ascending) order.  The frame call computes both on the device for every frame; a
// frame integration copies frame f's rows in instead of starting the two grid threads (INTEGRATION.md §5):
//
//     hvo_shim::fillGrid(&grid_counts[f * 3072], &grid_items[f * orb_capacity], mGrid);
//     hvo_shim::fillGrid(&lgrid_counts[f * 3072], &lgrid_items[f * line_grid_capacity], mGridForLine);
#ifndef HVO_SHIM_FRAMEGRIDGPU_H
#define HVO_SHIM_FRAMEGRIDGPU_H

#include <cstddef>
#include <cstdint>
#include <vector>

namespace hvo_shim {

// One frame's rows: counts [64 * 48] (cell = ix * 48 + iy), items = the cells' indices concatenated in cell order.  Every cell is
// replaced, so a grid that held an earlier frame's features is reused as is.
inline void fillGrid(const uint16_t* counts, const uint16_t* items, std::vector<std::size_t> (&grid)[64][48]) {
    std::size_t o = 0;
    for (int ix = 0; ix < 64; ++ix)
        for (int iy = 0; iy < 48; ++iy) {
            const std::size_t c = counts[ix * 48 + iy];
            grid[ix][iy].assign(items + o, items + o + c);
            o += c;
        }
}

}  // namespace hvo_shim

#endif
