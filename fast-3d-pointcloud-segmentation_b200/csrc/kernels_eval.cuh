// kernels_eval.cuh -- "next" row f1 of SURVEY.md section 8: Clustering::all_thresh (/root/reference/src/clustering.cpp:691-729)
// + the counting part of Testing (src/testing.cpp:62-146) from ONE merge replay.
// The reference re-clusters and re-intersects point sets for each of its 41 thresholds; continuing `cluster(state, t)` is the
// same as never having stopped, so every threshold is a PREFIX of one merge log (SURVEY.md CS4).  On the device:
//   merge log -> per-supervoxel segment labels at every threshold (the level tables of kernels_levels.cuh: dense labels in
//   ascending label order, as get_labeled_cloud :640-663); contingency table = histogram over the labelled voxel cloud of
//   (segment, truth label).
// Intersections by exact xyz (Testing::count_intersect) become equality of the voxel index: both clouds are voxel
// centroids of the same grid.
#pragma once
#include "kernels_merge.cuh"
#include "kernels_levels.cuh"

namespace f3ps {

// histogram over the labelled voxel cloud: position i belongs to initial supervoxel pos_run[i] and is voxel order[i]; its
// segment at level k is seg[s][k] (kernels_levels.cuh).  A phantom leaf counts twice, as it appears in the labelled cloud.
__global__ void __launch_bounds__(256) eval_table_kernel(const unsigned* __restrict__ pos_run, const unsigned* __restrict__ order, unsigned n_pos,
        const unsigned* __restrict__ seg, int Lp, int k, const unsigned* __restrict__ truth_dense, unsigned n_truth, unsigned* __restrict__ table) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pos; i += gridDim.x * blockDim.x) {
        const unsigned s = pos_run[i];
        if (s == 0xffffffffu) continue;                      // unowned voxel: absent from the segmentation
        const unsigned v = order ? order[i] : i;
        atomicAdd(&table[(size_t)seg[(size_t)s * Lp + k] * n_truth + truth_dense[v]], 1u);
    }
}

// contingency histogram of (segment, ground-truth label) pairs (Testing::compute_intersections, src/testing.cpp:88-146)
__global__ void __launch_bounds__(256) eval_pairs_kernel(const unsigned* __restrict__ seg, const unsigned* __restrict__ truth, long long n,
        unsigned n_cols, unsigned* __restrict__ table) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        atomicAdd(&table[(size_t)seg[i] * n_cols + truth[i]], 1u);
}

} // namespace f3ps
