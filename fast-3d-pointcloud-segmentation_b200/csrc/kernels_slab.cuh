// kernels_slab.cuh -- slab mode (SURVEY.md section 8e, row 2): one very large cloud cut into spatial slabs, one
// slab per GPU.  A slab is a contiguous range of the x-major Morton key (= a union of adjacency-octree subtrees),
// so a rank's voxels are a contiguous range of PCL's leaf index and every ordered sum of the single-GPU path
// (VoxelData::addPoint in input order, SupervoxelHelper::updateCentroid in idx order) keeps its order.
//
// The kernels here are the per-rank pieces between the exchanges; the exchanges themselves (NCCL all-reduce of
// the bounding box / key histogram, all-to-all of the points, all-gather of voxel / normal slices) are issued
// by the host driver on the same stream (f3ps/slab.py).
#pragma once
#include "kernels_vccs.cuh"

namespace f3ps {

constexpr int kSlabMaxWorld = 16;
constexpr int kSlabHistBitsMax = 15;

struct SlabSplitters { unsigned long long key[kSlabMaxWorld]; int n; };   // n = world - 1 ascending Morton keys

// histogram of the top bits of the Morton keys of this rank's valid points (equal-count slab cuts)
template <typename KeyT>
__global__ void __launch_bounds__(256) slab_key_hist_kernel(const KeyT* __restrict__ keys, const unsigned* __restrict__ n_ptr, int shift,
                                                            unsigned bins, unsigned* __restrict__ hist) {
    const unsigned n = *n_ptr;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned b = (unsigned)((unsigned long long)keys[i] >> shift);
        atomicAdd(&hist[min(b, bins - 1u)], 1u);
    }
}

// destination rank of every valid point = number of splitters <= key; per-destination totals
template <typename KeyT>
__global__ void __launch_bounds__(256) slab_dest_kernel(const KeyT* __restrict__ keys, const unsigned* __restrict__ n_ptr, SlabSplitters sp,
                                                        unsigned* __restrict__ dest, unsigned* __restrict__ totals) {
    __shared__ unsigned s_tot[kSlabMaxWorld];
    if (threadIdx.x < kSlabMaxWorld) s_tot[threadIdx.x] = 0u;
    __syncthreads();
    const unsigned n = *n_ptr;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned long long k = (unsigned long long)keys[i];
        unsigned d = 0;
        for (int s = 0; s < sp.n; ++s) d += k >= sp.key[s] ? 1u : 0u;
        dest[i] = d;
        atomicAdd(&s_tot[d], 1u);
    }
    __syncthreads();
    if (threadIdx.x < kSlabMaxWorld && s_tot[threadIdx.x]) atomicAdd(&totals[threadIdx.x], s_tot[threadIdx.x]);
}

// packed 16-byte records {x, y, z (folded), rgba bits} in destination order, input order kept inside a destination
__global__ void __launch_bounds__(256) slab_pack_kernel(PointLoader pl, const unsigned* __restrict__ idx, const unsigned* __restrict__ n_ptr,
                                                        float4* __restrict__ out) {
    const unsigned n = *n_ptr;
    for (unsigned j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const unsigned i = idx[j];
        float4 p = pl.xyzw(i);
        p.w = __uint_as_float(pl.rgba(i, p));
        out[j] = p;
    }
}

} // namespace f3ps
