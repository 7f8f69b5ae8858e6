// Test driver: hvo_shim::fillGrid (shim/FrameGridGPU.h) turns one frame's grid rows of the frame call into the reference's
// std::vector<std::size_t> grid[64][48].  Host code only: runs without a GPU.
//   in.bin : int32 magic, nframes, cap ; then [n][3072] uint16 counts, [n][cap] uint16 items
//   out.bin: per frame [3072] int32 cell sizes, then the cells' entries in cell order as int32
#include <cstdint>
#include <cstdio>
#include <vector>

#include "FrameGridGPU.h"

static std::vector<std::size_t> grid[64][48];

int main(int argc, char** argv) {
    if (argc != 3) { std::fprintf(stderr, "usage: shim_grid_fill in.bin out.bin\n"); return 2; }
    FILE* fi = std::fopen(argv[1], "rb");
    FILE* fo = std::fopen(argv[2], "wb");
    if (!fi || !fo) return 2;
    int32_t hdr[3];
    if (std::fread(hdr, 4, 3, fi) != 3 || hdr[0] != 0x44495247) return 3;
    const int n = hdr[1], cap = hdr[2];
    std::vector<uint16_t> counts((size_t)n * 3072), items((size_t)n * cap);
    if (std::fread(counts.data(), 2, counts.size(), fi) != counts.size() || std::fread(items.data(), 2, items.size(), fi) != items.size()) return 4;
    std::fclose(fi);
    grid[5][7].assign(3, 99);   // fillGrid replaces whatever the cells held
    for (int f = 0; f < n; ++f) {
        hvo_shim::fillGrid(&counts[(size_t)f * 3072], &items[(size_t)f * cap], grid);
        for (int ix = 0; ix < 64; ++ix)
            for (int iy = 0; iy < 48; ++iy) { const int32_t c = (int32_t)grid[ix][iy].size(); std::fwrite(&c, 4, 1, fo); }
        for (int ix = 0; ix < 64; ++ix)
            for (int iy = 0; iy < 48; ++iy)
                for (std::size_t v : grid[ix][iy]) { const int32_t x = (int32_t)v; std::fwrite(&x, 4, 1, fo); }
    }
    std::fclose(fo);
    return 0;
}
