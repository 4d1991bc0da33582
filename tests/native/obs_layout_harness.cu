// CPU-only dump of the observation row layout the kernels and the host code use (ObsLayout, mate_b200/csrc/mate_common.cuh),
// for tests/test_obs_layout.py to compare with mate_b200/constants.py.  No CUDA call is made: runs without a GPU.
// Arguments: triples nc nt no.  One line per triple:
//   nc nt no | camera row block starts | target row block starts | affine partition
// where a row's block starts are 0, own state, the three entity lists in the row's order and the row width, and the end
// of each entity list is also recomputed from entry_offset of its last entry.
#include <cstdio>
#include <cstdlib>

#include "../../mate_b200/csrc/mate_common.cuh"

using namespace mate;

static void row(const ObsLayout& L, bool cam_row) {
    const int order[3] = {cam_row ? KIND_TARGET : KIND_CAMERA, KIND_OBSTACLE, cam_row ? KIND_CAMERA : KIND_TARGET};
    printf(" | 0 %d", ObsLayout::SELF);
    for (int kind : order) printf(" %d", L.block(cam_row, kind));
    printf(" %d", cam_row ? L.dc() : L.dt());
    for (int kind : order)
        printf(" %d", L.count(kind) > 0 ? L.entry_offset(cam_row, kind, L.count(kind) - 1) + ObsLayout::width(kind) : L.block(cam_row, kind));
}

int main(int argc, char** argv) {
    printf("fixed %d %d %d\n", ObsLayout::PRESERVED, ObsLayout::WAREHOUSE, ObsLayout::TGT_EMPTY);
    for (int i = 1; i + 2 < argc; i += 3) {
        const ObsLayout L{atoi(argv[i]), atoi(argv[i + 1]), atoi(argv[i + 2])};
        printf("%d %d %d", L.nc, L.nt, L.no);
        row(L, true);
        row(L, false);
        printf(" | %d %d %d %d %d %d %d\n", ObsLayout::AFF_PRES, ObsLayout::AFF_TSELF, ObsLayout::AFF_CSELF, ObsLayout::AFF_TGT,
               ObsLayout::AFF_OBS, ObsLayout::AFF_CAM, ObsLayout::AFF_COLS);
    }
    return 0;
}
