// bow.cu — the per-feature part of DBoW2's vocabulary-tree transform (Frame::ComputeBoW / KeyFrame::ComputeBoW).
//
// Reference (snt-arg/visual_sgraphs):
//   Frame::ComputeBoW / KeyFrame::ComputeBoW            orb_slam3/src/Frame.cc:882-889, orb_slam3/src/KeyFrame.cc:99-108
//     -> TemplatedVocabulary::transform(features, BowVector&, FeatureVector&, levelsup = 4)
//        orb_slam3/Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1139-1205 (loop over the features)
//     -> transform(feature, word_id, weight, nid, levelsup)   :1225-1265: walk down from the root; at every node take
//        the child with the smallest F::distance (strict '<': the first child wins ties) until a leaf is reached; the
//        node passed at level L - levelsup is the feature's FeatureVector node
//   FORB::distance                                       orb_slam3/Thirdparty/DBoW2/DBoW2/FORB.cpp:81-101 (256-bit Hamming)
//
// The walk of each feature is independent: one thread per descriptor, the tree (child lists + 32-byte node
// descriptors, 35 MB for the k=10, L=6 ORB vocabulary) stays resident in device memory / L2.  What is left for the host
// is the bookkeeping on <= N entries that the reference does in feature order with double arithmetic:
// BowVector::addWeight(word, weight), FeatureVector::addFeature(node, i) and the final L1 normalisation.
#include <vector>

#include "vsg_internal.cuh"

struct vsg_vocabulary {
    int device = 0;
    int nnodes = 0, levels = 0;
    int *child_ptr = nullptr, *child_idx = nullptr;
    uint4 *node_desc = nullptr;
};

namespace vsg {

__global__ void __launch_bounds__(128) bow_transform_kernel(const int *__restrict__ child_ptr,
                                                            const int *__restrict__ child_idx,
                                                            const uint4 *__restrict__ node_desc,
                                                            const uint4 *__restrict__ desc, int n, int nid_level,
                                                            int *__restrict__ leaf_out, int *__restrict__ nid_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint4 a0 = __ldg(desc + 2 * i), a1 = __ldg(desc + 2 * i + 1);
    int final_id = 0, current_level = 0, nid = 0;           // nid_level <= 0 -> root (:1236)
    int cb = __ldg(child_ptr), ce = __ldg(child_ptr + 1);
    while (cb < ce) {                                        // do { ... } while (!isLeaf()) — the root always has children
        ++current_level;
        int best = 1 << 30;
        for (int c = cb; c < ce; ++c) {
            const int id = __ldg(child_idx + c);
            const uint4 b0 = __ldg(node_desc + 2 * id), b1 = __ldg(node_desc + 2 * id + 1);
            const int d = __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) +
                          __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
            if (d < best) { best = d; final_id = id; }       // strict '<' (:1253)
        }
        if (current_level == nid_level) nid = final_id;      // :1260-1261
        cb = __ldg(child_ptr + final_id);
        ce = __ldg(child_ptr + final_id + 1);
    }
    leaf_out[i] = final_id;
    nid_out[i] = nid;
}

}  // namespace vsg

using namespace vsg;

extern "C" {

vsg_status vsg_vocabulary_create(vsg_matcher *m, int nnodes, const int32_t *child_ptr, const int32_t *child_idx,
                                 const uint8_t *node_descriptors, int levels, vsg_vocabulary **out) {
    if (!m || !out || nnodes < 1 || !child_ptr || !node_descriptors || levels < 1) return VSG_ERR_INVALID;
    const int nchild = child_ptr[nnodes];
    if (child_ptr[0] != 0 || nchild != nnodes - 1 || (nchild > 0 && !child_idx)) {
        set_error("vsg_vocabulary_create: child lists must cover every node but the root exactly once");
        return VSG_ERR_INVALID;
    }
    if (child_ptr[1] == 0) { set_error("vsg_vocabulary_create: the root has no children (empty vocabulary)"); return VSG_ERR_INVALID; }
    for (int i = 0; i < nnodes; ++i)
        if (child_ptr[i + 1] < child_ptr[i]) { set_error("vsg_vocabulary_create: child_ptr must be non-decreasing"); return VSG_ERR_INVALID; }
    for (int c = 0; c < nchild; ++c)
        if (child_idx[c] <= 0 || child_idx[c] >= nnodes) { set_error("vsg_vocabulary_create: child index out of range"); return VSG_ERR_INVALID; }
    CK(cudaSetDevice(m->device));
    vsg_vocabulary *v = new vsg_vocabulary();
    v->device = m->device; v->nnodes = nnodes; v->levels = levels;
    bool ok = cuda_ok(cudaMalloc(&v->child_ptr, (size_t)(nnodes + 1) * 4), "cudaMalloc") &&
              cuda_ok(cudaMalloc(&v->child_idx, (size_t)std::max(nchild, 1) * 4), "cudaMalloc") &&
              cuda_ok(cudaMalloc(&v->node_desc, (size_t)nnodes * 32), "cudaMalloc") &&
              cuda_ok(cudaMemcpy(v->child_ptr, child_ptr, (size_t)(nnodes + 1) * 4, cudaMemcpyHostToDevice), "H2D") &&
              cuda_ok(cudaMemcpy(v->child_idx, child_idx, (size_t)nchild * 4, cudaMemcpyHostToDevice), "H2D") &&
              cuda_ok(cudaMemcpy(v->node_desc, node_descriptors, (size_t)nnodes * 32, cudaMemcpyHostToDevice), "H2D");
    if (!ok) { vsg_vocabulary_destroy(v); return VSG_ERR_CUDA; }
    *out = v;
    return VSG_OK;
}

void vsg_vocabulary_destroy(vsg_vocabulary *v) {
    if (!v) return;
    cudaSetDevice(v->device);
    cudaFree(v->child_ptr); cudaFree(v->child_idx); cudaFree(v->node_desc);
    delete v;
}

vsg_status vsg_bow_transform(vsg_matcher *m, const vsg_vocabulary *voc, const uint8_t *descriptors, int n, int levelsup,
                             int32_t *leaf_node_out, int32_t *feature_node_out) {
    if (!m || !voc || n < 0 || (n > 0 && (!descriptors || !leaf_node_out || !feature_node_out))) return VSG_ERR_INVALID;
    if (voc->device != m->device) { set_error("vsg_bow_transform: vocabulary lives on another device"); return VSG_ERR_INVALID; }
    if (n == 0) return VSG_OK;
    CK(cudaSetDevice(m->device));
    vsg_status st;
    if ((st = matcher_ensure(m, kSlotArg1, (size_t)n * 32)) || (st = matcher_ensure(m, kSlotOut, (size_t)n * 8))) return st;
    cudaStream_t s = m->stream;
    CK(cudaMemcpyAsync(m->buf[kSlotArg1], descriptors, (size_t)n * 32, cudaMemcpyHostToDevice, s));
    int *leaf = (int *)m->buf[kSlotOut], *nid = leaf + n;
    bow_transform_kernel<<<(n + 127) / 128, 128, 0, s>>>(voc->child_ptr, voc->child_idx, voc->node_desc,
                                                        (const uint4 *)m->buf[kSlotArg1], n, voc->levels - levelsup, leaf, nid);
    count_launch();
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(leaf_node_out, leaf, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(feature_node_out, nid, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VSG_OK;
}

}  // extern "C"
