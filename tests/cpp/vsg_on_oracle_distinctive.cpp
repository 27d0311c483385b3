// vsg_on_oracle_distinctive.cpp — TEST ADAPTER, linked beside tests/cpp/vsg_on_oracle.cpp: vsg_distinctive_descriptors on
// the CPU oracle port, by its definition in include/vsg_cuda.h (MapPoint::ComputeDistinctiveDescriptors' choice, once per
// point).  It lets tests/cpp/distinctive_batch_test.cpp run the shim's batched ComputeDistinctiveDescriptors(vpMPs) without
// a GPU.  Never linked into the product.
#include <cstddef>

#include "../../include/vsg_cuda.h"
#include "../../oracle/oracle.h"

extern "C" vsg_status vsg_distinctive_descriptors(vsg_matcher *, const uint8_t *descriptors, const int32_t *ptr, int npoints,
                                                  int32_t *best_out) {
    for (int p = 0; p < npoints; ++p)
        best_out[p] = orc_distinctive_descriptor(descriptors + (size_t)ptr[p] * 32, ptr[p + 1] - ptr[p]);
    return VSG_OK;
}
