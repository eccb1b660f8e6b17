// The block plan of one edge set (gnnb_prop_tc.cu builds it) as the tensor-core propagation kernels read it: the stand-alone
// gather-GEMM k_tc_prop (gnnb_prop_tc.cu) and the fused propagation + node-update kernel k_tc_fused (gnnb_tc.cu).
#pragma once

#include "gnnb_common.cuh"

namespace gnnb {

// A tile's K dimension (the sorted input slots its 128 output rows touch) is cut into K steps of 16 rows; a tile has at
// least one step.  The steps of a tile are contiguous in ks_rows and ks_w.
struct PropPlanDev {
    const int32_t* tile_ks0;      // [ntiles + 1] first K step of each tile
    const int32_t* ks_rows;       // [nksteps][16] input slot of each K row, -1 = zero row
    const uint16_t* ks_w;         // [nksteps] 8 KB weight blocks: [hi plane 4 KB][lo plane 4 KB], each 128 x 16 fp16 K-major without
                                  // swizzle, "piece-major": the 16-byte piece p (K 8p .. 8p + 7) of row m at p * 2048 + m * 16
    int ntiles;                   // tiles of the output layer = its slots / 128
    int nslots_in, nslots_out;    // rows per subdomain of the input / output layer (slot order, gnnb_common.cuh)
};

struct PropPlan;
const PropPlanDev& prop_plan_dev(const PropPlan* p);
double prop_plan_ksteps_per_tile(const PropPlan* p);

}  // namespace gnnb
