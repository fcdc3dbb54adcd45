// kernels_levels.cuh -- segmentation levels: the labels of several thresholds from ONE merge replay (f3ps_merge_levels).
// Every threshold is a prefix of the replay (SURVEY.md CS4): level k is the state after the first m_k merges, m_k = the first
// log index whose head weight is not below t_k.  On the device, with no host round trip between the stages:
//   forest  merge i makes rank(b) a child of rank(a) at time i (parent, when per initial supervoxel)
//   prefix  m_k per level (head weights are not monotone: a min-reduction, not a binary search)
//   dense   one block per level: dense label of every root alive after m_k merges, ascending rank = ascending label
//   roots   one thread per supervoxel walks the levels in ascending order, each walk continuing from the previous root
//           (a root at m_k is an ancestor of the one at m_{k-1}): seg[s][k] = dense label of s's region at level k
//   voxels  positions -> voxel table [V][Lp] with the owner rule of labeled_cloud_batch_kernel (a phantom leaf keeps its owner's)
//   points  out[k][p] = table[point_voxel[p]][k], the HBM-bound gather
// f3ps_eval_thresholds uses the first four stages for its contingency tables.
#pragma once
#include "common.cuh"

namespace f3ps {

constexpr int kMaxLevels = 256;
// row length of the per-supervoxel and per-voxel tables: one level as is, else padded to whole uint4s
inline int level_row(int L) { return L == 1 ? 1 : (L + 3) & ~3; }

__device__ __forceinline__ unsigned rank_of(const unsigned* __restrict__ sv_label, unsigned S, unsigned label) {
    unsigned lo = 0, hi = S;                     // sv_label ascends
    while (lo < hi) { const unsigned mid = (lo + hi) >> 1; if (sv_label[mid] < label) lo = mid + 1; else hi = mid; }
    return lo;
}

// when[] must hold 0xffffffff (never merged) before the launch
__global__ void __launch_bounds__(256) levels_forest_kernel(const unsigned* __restrict__ log_a, const unsigned* __restrict__ log_b, unsigned M,
        const unsigned* __restrict__ sv_label, unsigned S, unsigned* __restrict__ parent, unsigned* __restrict__ when) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < M; i += gridDim.x * blockDim.x) {
        const unsigned rb = rank_of(sv_label, S, log_b[i]);
        parent[rb] = rank_of(sv_label, S, log_a[i]); when[rb] = i;
    }
}

// one block, 2 * L words of dynamic shared memory.  Thresholds ascend, so the levels whose test !(w < t_k) log entry i passes
// are a prefix 0..c-1 of them; the first entry of each c, then a suffix minimum, gives m_k.
__global__ void __launch_bounds__(1024) levels_prefix_kernel(const float* __restrict__ w, unsigned M, const float* __restrict__ thr, int L,
        unsigned* __restrict__ m_out) {
    extern __shared__ unsigned s_lv[];
    float* s_t = reinterpret_cast<float*>(s_lv + L);
    for (int k = threadIdx.x; k < L; k += blockDim.x) { s_lv[k] = M; s_t[k] = thr[k]; }
    __syncthreads();
    for (unsigned i = threadIdx.x; i < M; i += blockDim.x) {
        const float x = w[i];
        int c = L;
        if (x == x) {                            // a NaN head weight stops every level
            int lo = 0, hi = L;                  // number of thresholds <= x
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_t[mid] <= x) lo = mid + 1; else hi = mid; }
            c = lo;
        }
        if (c > 0) atomicMin(&s_lv[c - 1], i);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned m = M;
        for (int k = L - 1; k >= 0; --k) { m = min(m, s_lv[k]); m_out[k] = m; }
    }
}

// one block per level: alive flags after m_k merges -> dense label per alive root (exclusive scan in ascending rank)
__global__ void __launch_bounds__(1024) levels_dense_kernel(const unsigned* __restrict__ when, unsigned S, const unsigned* __restrict__ m_lv,
        unsigned* __restrict__ dense, unsigned* __restrict__ n_segments) {
    __shared__ unsigned s_w[32]; __shared__ unsigned s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned m = m_lv[blockIdx.x];
    dense += (size_t)blockIdx.x * S;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (unsigned base = 0; base < S; base += blockDim.x) {
        const unsigned s = base + threadIdx.x;
        const unsigned alive = (s < S && when[s] >= m) ? 1u : 0u;
        unsigned v = alive;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(kFull, v, o); if (lane >= o) v += t; }
        if (lane == 31) s_w[warp] = v;
        __syncthreads();
        unsigned wb = 0;
        for (int w = 0; w < warp; ++w) wb += s_w[w];
        const unsigned carry = s_carry;
        if (s < S) dense[s] = alive ? carry + wb + v - 1u : 0xffffffffu;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) s_carry = carry + wb + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) n_segments[blockIdx.x] = s_carry;
}

// seg[s][k] (row length Lp): dense label at level k of the region that holds initial supervoxel s; padding = 0xffffffff
__global__ void __launch_bounds__(256) levels_roots_kernel(const unsigned* __restrict__ parent, const unsigned* __restrict__ when,
        const unsigned* __restrict__ m_lv, const unsigned* __restrict__ dense, unsigned S, int L, int Lp, unsigned* __restrict__ seg) {
    for (unsigned s = blockIdx.x * blockDim.x + threadIdx.x; s < S; s += gridDim.x * blockDim.x) {
        unsigned r = s;
        for (int k = 0; k < L; ++k) {
            const unsigned m = m_lv[k];
            while (when[r] < m) r = parent[r];
            seg[(size_t)s * Lp + k] = dense[(size_t)k * S + r];
        }
        for (int k = L; k < Lp; ++k) seg[(size_t)s * Lp + k] = 0xffffffffu;
    }
}

// positions -> voxel rows: position i belongs to initial supervoxel pos_run[i] and is voxel vox_of_pos[i].  A phantom leaf's
// position (its run's label is not the voxel's owner) leaves the row to the owner's position; unowned voxels keep 0xffffffff.
__global__ void __launch_bounds__(256) levels_voxel_kernel(const unsigned* __restrict__ pos_run, unsigned n_pos, const unsigned* __restrict__ vox_of_pos,
        const unsigned* __restrict__ pos_label, const unsigned* __restrict__ owner, const unsigned* __restrict__ seg, int Lp, unsigned* __restrict__ table) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pos; i += gridDim.x * blockDim.x) {
        const unsigned s = pos_run[i];
        if (s == 0xffffffffu) continue;
        const unsigned v = vox_of_pos[i];
        if (owner && owner[v] != pos_label[i]) continue;
        if (Lp == 1) { table[v] = seg[s]; continue; }
        const uint4* src = reinterpret_cast<const uint4*>(seg + (size_t)s * Lp);
        uint4* dst = reinterpret_cast<uint4*>(table + (size_t)v * Lp);
        for (int q = 0; q < Lp / 4; ++q) dst[q] = src[q];
    }
}

// out[k][p] = table[pv[p]][k] (0xffffffff for a point without a voxel; pv == nullptr: row first + p): four points per thread.
// pv comes in as one int4, each point's row as uint4s (Lp % 4 == 0) or one word (Lp == 1); a 4x4 register transpose turns them
// into one uint4 store per level row.  vec_out: every output row starts 16-byte aligned (aligned base, N % 4 == 0).  Loads and
// stores stream past L1 and are evicted first from L2, so the table stays L2-resident.
__global__ void __launch_bounds__(256) level_point_labels_kernel(const int* __restrict__ pv, int first, long long N, const unsigned* __restrict__ table,
        int L, int Lp, unsigned* __restrict__ out, int vec_out) {
    const long long groups = (N + 3) >> 2;
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < groups; g += (long long)gridDim.x * blockDim.x) {
        const long long p0 = g << 2;
        int v[4];
        if (!pv) for (int j = 0; j < 4; ++j) v[j] = p0 + j < N ? first + (int)(p0 + j) : -1;
        else if (p0 + 3 < N) { const int4 q = __ldcs(reinterpret_cast<const int4*>(pv) + g); v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w; }
        else for (int j = 0; j < 4; ++j) v[j] = p0 + j < N ? pv[p0 + j] : -1;
        const bool full = vec_out && p0 + 3 < N;
        for (int kc = 0; kc < L; kc += 4) {
            uint4 r[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (v[j] < 0) r[j] = make_uint4(kFull, kFull, kFull, kFull);
                else if (Lp == 1) r[j].x = __ldg(table + v[j]);
                else r[j] = __ldg(reinterpret_cast<const uint4*>(table + (size_t)v[j] * Lp + kc));
            }
            const int kn = min(4, L - kc);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                if (kk >= kn) break;
                const unsigned a = kk == 0 ? r[0].x : kk == 1 ? r[0].y : kk == 2 ? r[0].z : r[0].w;
                const unsigned b = kk == 0 ? r[1].x : kk == 1 ? r[1].y : kk == 2 ? r[1].z : r[1].w;
                const unsigned c = kk == 0 ? r[2].x : kk == 1 ? r[2].y : kk == 2 ? r[2].z : r[2].w;
                const unsigned d = kk == 0 ? r[3].x : kk == 1 ? r[3].y : kk == 2 ? r[3].z : r[3].w;
                unsigned* row = out + (size_t)(kc + kk) * N + p0;
                if (full) __stcs(reinterpret_cast<uint4*>(row), make_uint4(a, b, c, d));
                else {
                    const unsigned e[4] = {a, b, c, d};
                    for (int j = 0; j < 4 && p0 + j < N; ++j) __stcs(row + j, e[j]);
                }
            }
        }
    }
}

} // namespace f3ps
