// Manhattan::computeNormalsLPVO (csrc/lpvo.cu): the geometry, scratch and launch of the rows -> cols -> normals chain, shared by the
// standalone hvo_lpvo handle and the frame pipeline's LPVO stage (csrc/frame.cu).
#pragma once
#include "hvo_common.cuh"

namespace hvo {

struct LpvoGeom {
    int W, H, nsu, nsv;  // lattice: u = 10 + 15 j (j < nsu), v = 10 + 15 i (i < nsv)
    float cx, cy, inv_fx, inv_fy, factor;
};

LpvoGeom lpvo_geom(const hvo_plane_params& cam, int width, int height);
inline int lpvo_capacity(const LpvoGeom& g) { return g.nsu * g.nsv; }

// Row sums and lattice integrals of `frames` frames: the chain runs over sub-batches of at most that many frames.
struct LpvoScratch {
    int frames = 0;
    double* rowsum = nullptr;
    double* integ = nullptr;
};
int lpvo_scratch_alloc(const LpvoGeom& g, int frames, LpvoScratch* s);
void lpvo_scratch_free(LpvoScratch* s);

// n frames of raw depth (rows f * W * H) -> frame f's samples in rows f * capacity of the outputs; counts[f] of them.  Queued on s;
// adds the number of kernel launches to *launches.
int lpvo_launch(cudaStream_t s, const LpvoGeom& g, const LpvoScratch& sc, const uint16_t* d_depth, int n, double* d_normals3, float* d_z,
                int32_t* d_pix2, int32_t* d_counts, int* launches);

}  // namespace hvo
