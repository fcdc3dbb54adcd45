// kernels_segments.cuh -- segment extraction (f3ps_get_segment_points / _voxels / _info): the points or voxels of every segment of
// one level, grouped, and one descriptor per segment.  On the level tables of kernels_levels.cuh:
//   keys     SegmentKeyOp (compact_kernel): (label, index) of every point / voxel with a segment at the level, in index order
//   sort     sort_pairs<unsigned> on the label (stable LSD), so the indices inside a segment stay ascending
//   offsets  K-bin count over the sorted labels, then an exclusive scan into offsets[K+1] (and the chunk offsets below)
//   partials one block per chunk of kSegChunk CSR positions of one segment: fixed tree reduction of its points
//   info     one warp per segment folds its chunk partials in chunk order
// Every sum has a fixed shape that depends only on the CSR, never on the grid or on timing: no float atomics, the same bits
// from every call.
#pragma once
#include "../../include/f3ps.h"
#include "common.cuh"
#include "kernels_vccs.cuh"

namespace f3ps {

constexpr int kSegChunk = 4096;             // CSR positions per partial
constexpr int kSegThreads = 256;            // threads per partial block: kSegChunk / kSegThreads points per thread
constexpr int kSegRun = 16;                 // sorted labels per thread of the count kernel

// (label at `level`, index) of every point (pv: its voxel, -1 = none) or voxel (pv == nullptr) that a segment holds
struct SegmentKeyOp {
    const int* pv; const unsigned* lv_vox; int Lp; int level; unsigned* keys; unsigned* vals;
    typedef unsigned Payload;
    __device__ __forceinline__ bool test(int64_t i, Payload& lab) const {
        const int v = pv ? pv[i] : (int)i;
        if (v < 0) return false;
        lab = lv_vox[(size_t)v * Lp + level];
        return lab != kFull;
    }
    __device__ __forceinline__ void emit(unsigned pos, int64_t i, const Payload& lab) const { keys[pos] = lab; vals[pos] = (unsigned)i; }
};

// counts[key] over n_ptr[0] keys (counts zeroed before); one atomic per run of equal keys inside a thread's kSegRun keys
__global__ void __launch_bounds__(256) segment_count_kernel(const unsigned* __restrict__ keys, const unsigned* __restrict__ n_ptr,
                                                            unsigned* __restrict__ counts) {
    const unsigned n = *n_ptr;
    for (unsigned c = blockIdx.x * blockDim.x + threadIdx.x; (size_t)c * kSegRun < n; c += gridDim.x * blockDim.x) {
        const unsigned i0 = c * kSegRun, i1 = min(n, i0 + kSegRun);
        unsigned cur = keys[i0], run = 0;
        for (unsigned i = i0; i < i1; ++i) {
            const unsigned k = keys[i];
            if (k != cur) { atomicAdd(&counts[cur], run); cur = k; run = 0; }
            ++run;
        }
        atomicAdd(&counts[cur], run);
    }
}

// exclusive block-wide scan of one value per thread (blockDim.x a multiple of 32, s_w: 32 words); *total = the block's sum
template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T* s_w, T& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    T x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const T t = __shfl_up_sync(kFull, x, o); if (lane >= o) x += t; }
    if (lane == 31) s_w[warp] = x;
    __syncthreads();
    T wb = 0; total = 0;
    for (int w = 0; w < nw; ++w) { const T c = s_w[w]; if (w < warp) wb += c; total += c; }
    __syncthreads();
    return wb + x - v;
}

// one block: offsets[K+1] = exclusive scan of counts (a segment without members gets an empty range), chunk_off[K+1] = the same
// over ceil(counts / kSegChunk), the partials of each segment
__global__ void __launch_bounds__(1024) segment_offsets_kernel(const unsigned* __restrict__ counts, unsigned K, long long* __restrict__ offsets,
                                                               unsigned* __restrict__ chunk_off) {
    __shared__ long long s_a[32]; __shared__ unsigned s_b[32];
    long long carry_a = 0; unsigned carry_b = 0;
    for (unsigned base = 0; base < K; base += blockDim.x) {
        const unsigned j = base + threadIdx.x;
        const unsigned c = j < K ? counts[j] : 0u;
        long long ta; unsigned tb;
        const long long ea = block_exclusive_scan<long long>((long long)c, s_a, ta);
        const unsigned eb = block_exclusive_scan<unsigned>((c + kSegChunk - 1) / kSegChunk, s_b, tb);
        if (j < K) { offsets[j] = carry_a + ea; chunk_off[j] = carry_b + eb; }
        carry_a += ta; carry_b += tb;
    }
    if (threadIdx.x == 0) { offsets[K] = carry_a; chunk_off[K] = carry_b; }
}

struct SegPartial {                          // 64 bytes
    double sum[3];                           // xyz sums
    float mn[3], mx[3];
    unsigned rgb[3];                         // r, g, b sums (a chunk: at most kSegChunk * 255)
    unsigned pad;
};

// one block per chunk: chunk c is chunk c - chunk_off[j] of segment j (the last j with chunk_off[j] <= c).  Thread t reduces the
// positions t, t + 256, ... of the chunk in order, then a fixed xor-shuffle tree per warp and warp 0 over the warps in order.
__global__ void __launch_bounds__(kSegThreads) segment_partials_kernel(PointLoader pl, const unsigned* __restrict__ index,
        const long long* __restrict__ offsets, const unsigned* __restrict__ chunk_off, unsigned K, SegPartial* __restrict__ part) {
    __shared__ SegPartial s_p[kSegThreads / 32];
    const unsigned c = blockIdx.x;
    if (c >= chunk_off[K]) return;
    unsigned lo = 0, hi = K - 1;
    while (lo < hi) { const unsigned mid = (lo + hi + 1) >> 1; if (chunk_off[mid] <= c) lo = mid; else hi = mid - 1; }
    const long long b = offsets[lo] + (long long)(c - chunk_off[lo]) * kSegChunk;
    const long long e = min(offsets[lo + 1], b + kSegChunk);
    double s[3] = {0.0, 0.0, 0.0};
    float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    unsigned rgb[3] = {0u, 0u, 0u};
#pragma unroll 4
    for (int q = 0; q < kSegChunk / kSegThreads; ++q) {
        const long long p = b + q * kSegThreads + threadIdx.x;
        if (p >= e) break;
        const unsigned i = __ldcs(index + p);
        const float4 x = pl.xyzw(i);
        const uint32_t col = pl.rgba(i, x);
        s[0] += (double)x.x; s[1] += (double)x.y; s[2] += (double)x.z;
        mn[0] = fminf(mn[0], x.x); mn[1] = fminf(mn[1], x.y); mn[2] = fminf(mn[2], x.z);
        mx[0] = fmaxf(mx[0], x.x); mx[1] = fmaxf(mx[1], x.y); mx[2] = fmaxf(mx[2], x.z);
        rgb[0] += (col >> 16) & 255u; rgb[1] += (col >> 8) & 255u; rgb[2] += col & 255u;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            s[a] += __shfl_xor_sync(kFull, s[a], o);
            mn[a] = fminf(mn[a], __shfl_xor_sync(kFull, mn[a], o));
            mx[a] = fmaxf(mx[a], __shfl_xor_sync(kFull, mx[a], o));
            rgb[a] += __shfl_xor_sync(kFull, rgb[a], o);
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        SegPartial& w = s_p[warp];
        for (int a = 0; a < 3; ++a) { w.sum[a] = s[a]; w.mn[a] = mn[a]; w.mx[a] = mx[a]; w.rgb[a] = rgb[a]; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        SegPartial r = s_p[0];
        for (int w = 1; w < kSegThreads / 32; ++w)
            for (int a = 0; a < 3; ++a) {
                r.sum[a] += s_p[w].sum[a]; r.mn[a] = fminf(r.mn[a], s_p[w].mn[a]); r.mx[a] = fmaxf(r.mx[a], s_p[w].mx[a]); r.rgb[a] += s_p[w].rgb[a];
            }
        r.pad = 0;
        part[c] = r;
    }
}

// one warp per segment: the lanes load 32 partials at a time, every lane folds them in chunk order.  n_points from the point
// offsets, n_voxels from the voxel offsets; a segment without points gets NaN bounds, centroid and colour.  region_label is
// written by segment_region_kernel.
__global__ void __launch_bounds__(256) segment_info_kernel(const SegPartial* __restrict__ part, const unsigned* __restrict__ chunk_off,
        const long long* __restrict__ offsets, const long long* __restrict__ vox_offsets, unsigned K, f3ps_segment_info* __restrict__ out) {
    const unsigned lane = threadIdx.x & 31;
    const unsigned j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (j >= K) return;
    const unsigned c0 = chunk_off[j], c1 = chunk_off[j + 1];
    double s[3] = {0.0, 0.0, 0.0};
    float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    unsigned long long rgb[3] = {0ull, 0ull, 0ull};
    for (unsigned base = c0; base < c1; base += 32) {
        SegPartial p{};
        if (base + lane < c1) p = part[base + lane];
        const unsigned nq = min(32u, c1 - base);
        for (unsigned q = 0; q < nq; ++q) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                s[a] += __shfl_sync(kFull, p.sum[a], q);
                mn[a] = fminf(mn[a], __shfl_sync(kFull, p.mn[a], q));
                mx[a] = fmaxf(mx[a], __shfl_sync(kFull, p.mx[a], q));
                rgb[a] += __shfl_sync(kFull, p.rgb[a], q);
            }
        }
    }
    if (lane) return;
    const long long n = offsets[j + 1] - offsets[j];
    f3ps_segment_info r;
    r.region_label = 0xffffffffu;
    r.n_voxels = (int32_t)(vox_offsets[j + 1] - vox_offsets[j]);
    r.n_points = n;
    const float nan = __int_as_float(0x7fc00000);
    for (int a = 0; a < 3; ++a) {
        r.min_xyz[a] = n ? mn[a] : nan; r.max_xyz[a] = n ? mx[a] : nan;
        r.centroid[a] = n ? (float)(s[a] / (double)n) : nan;
        r.mean_rgb[a] = n ? (float)((double)rgb[a] / (double)n) : nan;
    }
    out[j] = r;
}

// region_label of every segment: the label of its root, the initial supervoxel whose dense label at the level it is
__global__ void __launch_bounds__(256) segment_region_kernel(const unsigned* __restrict__ dense, const unsigned* __restrict__ sv_label, unsigned S,
                                                             f3ps_segment_info* __restrict__ out) {
    for (unsigned s = blockIdx.x * blockDim.x + threadIdx.x; s < S; s += gridDim.x * blockDim.x) {
        const unsigned d = dense[s];
        if (d != kFull) out[d].region_label = sv_label[s];
    }
}

} // namespace f3ps
