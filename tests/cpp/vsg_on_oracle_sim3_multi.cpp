// vsg_on_oracle_sim3_multi.cpp — TEST ADAPTER, linked beside tests/cpp/vsg_on_oracle.cpp: vsg_fuse_search_sim3_multi on the
// CPU oracle port, by its definition in include/vsg_cuda.h (vsg_fuse_search, variant 1, once per target).  It lets
// tests/cpp/search_and_fuse_test.cpp run the shim's batched Fuse(vpKFs, vScw, vpPoints, th) without a GPU.  Never linked
// into the product.
#include <cstddef>

#include "../../include/vsg_cuda.h"

extern "C" vsg_status vsg_fuse_search_sim3_multi(vsg_matcher *m, int ntargets, const vsg_frame *const *KFs, int n,
                                                 const vsg_search_point *pts, const uint8_t *desc, float th, int32_t *best_idx_out) {
    for (int t = 0; t < ntargets; ++t) {
        const vsg_status st = vsg_fuse_search(m, KFs[t], n, pts + (size_t)t * n, desc, th, nullptr, 1, best_idx_out + (size_t)t * n,
                                              nullptr);
        if (st != VSG_OK) return st;
    }
    return VSG_OK;
}
