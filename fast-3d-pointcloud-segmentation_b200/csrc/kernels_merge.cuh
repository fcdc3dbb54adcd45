// kernels_merge.cuh -- K7: the greedy hierarchical merge, Clustering::cluster / merge / contains
// (/root/reference/src/clustering.cpp:384-469, 497-506), as ONE persistent thread block that
// replays the reference's serial min-edge order exactly (SURVEY.md Appendix C):
//   * multimap order  ==  argmin over (weight, stamp)   -- stamp rule C.2
//   * region statistics are continued, not recomputed     -- prefix property C.3
// Per merge: block-wide argmin -> [warp 0: fold region b onto a, eigen-solve the new normal]
// in parallel with [warps 1..31: collect the edges incident to a or b] -> order them by their old
// key, drop duplicates (the earlier survives), recompute the survivors' weights in parallel
// (CIEDE2000 in FP64), assign tie stamps.
#pragma once
#include "kernels_graph.cuh"

namespace f3ps {

constexpr int kMergeThreads = 1024;
struct MergeSortRec { float w; unsigned slot; long long st; };      // old key of a touched edge + where it sits in the unsorted list
struct MergeScratch { int* e[2]; float* w[2]; long long* st[2]; unsigned* x[2]; unsigned char* cls; unsigned* mark; MergeSortRec* sortbuf; };
constexpr int kMergeSortSmem = 8192;   // records sorted in (dynamic) shared memory; longer lists sort in the global buffer

struct MergeLog { unsigned* a; unsigned* b; float* w; unsigned* edges_left; unsigned* regions_left; };
struct MergeCtl {
    unsigned n_merges, edges_alive, regions_alive, error;
    unsigned nan_weights, max_touched, pad0, pad1;
    long long counter;
    unsigned long long fold_steps;
    unsigned long long phase_cycles[32];  // clock64 deltas / event counts per phase (see f3ps_merge_profile)
};

__device__ __forceinline__ bool key_less(float w1, long long s1, float w2, long long s2) {
    return w1 < w2 || (w1 == w2 && s1 < s2);
}

// Ordered fold of region b's rope (its runs of position-ordered voxels) onto a region, one accumulator chain per lane, the
// same scalar sequence as stats_step (src/color_utilities.cpp:130-134 + computeMeanAndCovarianceMatrix).
//   COLOUR == false: lanes 0..8 hold the nine raw sums (xx,xy,xz,yy,yz,zz,x,y,z)
//   COLOUR == true : lanes 0..2 hold the running means r,g,b; the reciprocals 1/k of a chunk are prepared by all lanes at once
// Chunks of <= 64 voxels: while the chains walk chunk i out of shared memory, the loads of chunk i+1 (and the bounds of the
// run after it) are in flight.  `cnt` = voxels folded so far as float; requires cnt + |b| < 2^24 (exact integer floats).
template <bool COLOUR>
__device__ __forceinline__ unsigned fold_rope_lanes(float& v, float& cnt, const RegionArrays& R, unsigned b, const unsigned* __restrict__ run_start,
        const unsigned* __restrict__ run_end, const float4* __restrict__ pos_data, float* __restrict__ stage, int lane) {
    constexpr int RS = COLOUR ? 4 : 9;
    int run = R.head[b];
    unsigned rs = run_start[run], re = run_end[run];
    int nxt = R.next_run[run];
    unsigned nrs = 0, nre = 0; int nnxt = -1;
    if (nxt >= 0) { nrs = run_start[nxt]; nre = run_end[nxt]; nnxt = R.next_run[nxt]; }
    unsigned cs = rs, ce = min(rs + 64u, re), steps = 0;
    float4 p[2], q[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) if (cs + 32u * h + lane < ce) p[h] = __ldcg(pos_data + cs + 32u * h + lane);
    while (true) {
        // the chunk after this one
        bool have_next = false; unsigned ns = 0, ne = 0;
        if (ce < re) { ns = ce; ne = min(ce + 64u, re); have_next = true; }
        else if (nxt >= 0) {
            run = nxt; rs = nrs; re = nre; nxt = nnxt;
            if (nxt >= 0) { nrs = run_start[nxt]; nre = run_end[nxt]; nnxt = R.next_run[nxt]; }
            ns = rs; ne = min(rs + 64u, re); have_next = true;
        }
        const unsigned m = ce - cs;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (cs + 32u * h + lane < ce) {
                float* row = stage + (32 * h + lane) * RS;
                if (COLOUR) {
                    const uint32_t c = __float_as_uint(p[h].w);
                    row[0] = (float)((c >> 16) & 255u); row[1] = (float)((c >> 8) & 255u); row[2] = (float)(c & 255u);
                    row[3] = 1 / (cnt + (float)(32 * h + lane + 1));
                } else {
                    row[0] = p[h].x * p[h].x; row[1] = p[h].x * p[h].y; row[2] = p[h].x * p[h].z; row[3] = p[h].y * p[h].y; row[4] = p[h].y * p[h].z;
                    row[5] = p[h].z * p[h].z; row[6] = p[h].x; row[7] = p[h].y; row[8] = p[h].z;
                }
            }
        }
        __syncwarp();
        if (have_next) {
#pragma unroll
            for (int h = 0; h < 2; ++h) if (ns + 32u * h + lane < ne) q[h] = __ldcg(pos_data + ns + 32u * h + lane);
        }
        if (COLOUR) {
            if (lane < 3) {
                unsigned j = 0;
                for (; j + 4 <= m; j += 4) {
                    const float x0 = stage[j * 4 + lane], x1 = stage[j * 4 + 4 + lane], x2 = stage[j * 4 + 8 + lane], x3 = stage[j * 4 + 12 + lane];
                    const float i0 = stage[j * 4 + 3], i1 = stage[j * 4 + 7], i2 = stage[j * 4 + 11], i3 = stage[j * 4 + 15];
                    v = v + i0 * (x0 - v); v = v + i1 * (x1 - v); v = v + i2 * (x2 - v); v = v + i3 * (x3 - v);
                }
                for (; j < m; ++j) v = v + stage[j * 4 + 3] * (stage[j * 4 + lane] - v);
            }
        } else {
            if (lane < 9) {
                unsigned j = 0;
                for (; j + 4 <= m; j += 4) {
                    const float x0 = stage[j * 9 + lane], x1 = stage[j * 9 + 9 + lane], x2 = stage[j * 9 + 18 + lane], x3 = stage[j * 9 + 27 + lane];
                    v += x0; v += x1; v += x2; v += x3;
                }
                for (; j < m; ++j) v += stage[j * 9 + lane];
            }
        }
        cnt += (float)m; steps += m;
        __syncwarp();
        if (!have_next) break;
        p[0] = q[0]; p[1] = q[1]; cs = ns; ce = ne;
    }
    return steps;
}

// Fallback fold (a region beyond 2^24 voxels, or no position-ordered voxel array): the whole statistics replicated in every
// lane.  Never inlined: it is off the hot path and must not occupy the merge loop's instruction footprint.
__device__ __noinline__ unsigned long long merge_fold_fallback(RegionArrays R, EdgeParams ep, unsigned a, unsigned b, const unsigned* __restrict__ run_start,
        const unsigned* __restrict__ run_end, const unsigned* __restrict__ order, const float4* __restrict__ vox_xyz, int lane) {
    RegionStats st; load_stats(R, (int)a, st);
    unsigned long long steps = 0;
    for (int run = R.head[b]; run >= 0; run = R.next_run[run]) {
        const unsigned rs = run_start[run], re = run_end[run];
        fold_run(st, order, rs, re, vox_xyz, lane);       // voxels_ = a ++ b  (:408)
        steps += re - rs;
    }
    if (lane == 0) {
        store_stats(R, (int)a, st);
        const float fn = (float)st.n;
        const float cx = st.accu[6] / fn, cy = st.accu[7] / fn, cz = st.accu[8] / fn;   // computeCentroid (:411-413)
        float n[3]; float curv;
        if (st.n < 3) { n[0] = n[1] = n[2] = nanf(""); curv = n[0]; }
        else plane_from_accu(st.accu, st.n, n, curv);                                     // computePointNormal (:415-417)
        flip_and_normalize(cx, cy, cz, n);                                                // :418-420
        R.centroid[a] = make_float4(cx, cy, cz, 0.0f);
        R.normal[a] = make_float4(n[0], n[1], n[2], curv);
        float cv[3]; colour_vector(ep, st.r, st.g, st.b, cv);
        R.cvec[a] = make_float4(cv[0], cv[1], cv[2], 0.0f);
    }
    return steps;
}

// packed endpoints of an edge for the incidence scan: 16 + 16 bits when the graph has < 65,536 regions, else 32 + 32
template <typename PK> struct PkOps;
template <> struct PkOps<unsigned> {
    static constexpr unsigned kDead = 0xffffffffu;
    static __device__ __forceinline__ unsigned pack(unsigned a, unsigned b) { return (a << 16) | b; }
    static __device__ __forceinline__ unsigned lo(unsigned p) { return p >> 16; }
    static __device__ __forceinline__ unsigned hi(unsigned p) { return p & 0xffffu; }
};
template <> struct PkOps<unsigned long long> {
    static constexpr unsigned long long kDead = ~0ull;
    static __device__ __forceinline__ unsigned long long pack(unsigned a, unsigned b) { return ((unsigned long long)a << 32) | b; }
    static __device__ __forceinline__ unsigned lo(unsigned long long p) { return (unsigned)(p >> 32); }
    static __device__ __forceinline__ unsigned hi(unsigned long long p) { return (unsigned)p; }
};

constexpr int kMergeTcap = 1024;       // touched edges of one merge handled in shared memory; more go through the global scratch

// The general kernel: any S, E, T; everything in global memory (L2-resident), one CTA.
//   head      : every thread caches the minimum of its own contiguous strip of edges and rescans the strip only after one of
//               its edges was re-weighted or died ("dirty"), so a merge costs O(T * E / 1024) loads instead of O(E)
//   incidence : one packed word per edge (16 + 16 or 32 + 32 bits), eight independent loads in flight per thread
//   ordering / dedupe / tie stamps of the <= 1024 touched edges in shared memory (ballot prefix counts for the stamps)
template <typename PK>
__global__ void __launch_bounds__(kMergeThreads, 1) merge_kernel(RegionArrays R, EdgeArrays E, const unsigned* __restrict__ n_edges_ptr,
        const unsigned* __restrict__ n_sv_ptr, EdgeParams ep, const float* __restrict__ lambda_dev, float threshold,
        const unsigned* __restrict__ run_start, const unsigned* __restrict__ run_end, const unsigned* __restrict__ order,
        const float4* __restrict__ vox_xyz, const unsigned* __restrict__ sv_label, MergeLog mlog, unsigned log_cap, MergeCtl* ctl, MergeScratch scr,
        PK* __restrict__ pk, const float4* __restrict__ pos_data) {
    typedef PkOps<PK> P;
    extern __shared__ __align__(16) unsigned char dyn_smem[];     // kMergeSortSmem sort records
    __shared__ float s_rw[32]; __shared__ long long s_rs[32]; __shared__ int s_ri[32];
    __shared__ int s_head; __shared__ float s_head_w;
    __shared__ int s_tcount;
    __shared__ int sm_e[2][kMergeTcap]; __shared__ float sm_w[2][kMergeTcap]; __shared__ long long sm_st[2][kMergeTcap];
    __shared__ unsigned sm_x[2][kMergeTcap]; __shared__ unsigned char sm_cls[kMergeTcap];
    __shared__ unsigned char s_dirty[kMergeThreads];
    __shared__ unsigned s_wb[32], s_wf[32], s_wd[32];
    __shared__ float s_stage[64 * 9]; __shared__ float s_stage2[64 * 4];
    __shared__ int s_lanes;
    __shared__ unsigned s_nm, s_ealive, s_ralive; __shared__ long long s_counter;
    __shared__ unsigned long long s_fold;
    __shared__ unsigned s_maxT;
    unsigned long long pc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long t_prev = clock64();
#undef PHASE
#define PHASE(i) do { if (tid == 0) { long long t_now = clock64(); pc[i] += (unsigned long long)(t_now - t_prev); t_prev = t_now; } } while (0)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned nE = *n_edges_ptr;
    if (lambda_dev) ep.lambda = *lambda_dev;
    if (tid == 0) { s_nm = 0; s_ealive = nE; s_ralive = *n_sv_ptr; s_counter = (long long)nE; s_fold = 0; s_maxT = 0; }
    const float INF = __int_as_float(0x7f800000);
    enum { C_KEEP = 0, C_FRONT = 1, C_BACK = 2, C_DUP = 3 };
    // strip of this thread and its cached minimum
    // thread (warp w, lane l) owns the edges w * 32 K + 32 j + l, j < K: a warp's strips interleave, so its rescans coalesce
    const unsigned K = max(1u, (nE + kMergeThreads - 1) / kMergeThreads), W = 32u * K;
    const unsigned my_base = (unsigned)warp * W + (unsigned)lane;
#define F3PS_OWNER(e) ((((unsigned)(e)) / W) * 32u + (((unsigned)(e)) & 31u))
    float cw = INF; long long cs = kDeadStamp; int ci = -1;
    s_dirty[tid] = 1;
    for (unsigned e = tid; e < nE; e += kMergeThreads) pk[e] = E.stamp[e] == kDeadStamp ? P::kDead : P::pack(E.a[e], E.b[e]);
    for (unsigned r = tid; r < *n_sv_ptr; r += kMergeThreads) scr.mark[r] = 0xffffffffu;
    __threadfence();
    __syncthreads();

    while (true) {
        // ---- A: head of the weight map = argmin (w, stamp) -------------------------------
        if (s_dirty[tid]) {
            s_dirty[tid] = 0;
            cw = INF; cs = kDeadStamp; ci = -1;
            for (unsigned j0 = 0; j0 < K; j0 += 8) {
                long long st[8]; float w[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const unsigned e = my_base + (j0 + k) * 32u;
                    const bool in = j0 + k < K && e < nE;
                    st[k] = in ? __ldcg(E.stamp + e) : kDeadStamp;
                    w[k] = in ? __ldcg(E.w + e) : INF;
                }
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if (st[k] != kDeadStamp && (ci < 0 || key_less(w[k], st[k], cw, cs))) { cw = w[k]; cs = st[k]; ci = (int)(my_base + (j0 + k) * 32u); }
            }
        }
        float bw = cw; long long bs = cs; int bi = ci;
#pragma unroll
        for (int off = 16; off; off >>= 1) {
            const float ow = __shfl_xor_sync(kFull, bw, off); const long long os = __shfl_xor_sync(kFull, bs, off);
            const int oi = __shfl_xor_sync(kFull, bi, off);
            if (oi >= 0 && (bi < 0 || key_less(ow, os, bw, bs))) { bw = ow; bs = os; bi = oi; }
        }
        if (lane == 0) { s_rw[warp] = bw; s_rs[warp] = bs; s_ri[warp] = bi; }
        __syncthreads();
        if (warp == 0) {
            bw = s_rw[lane]; bs = s_rs[lane]; bi = s_ri[lane];
#pragma unroll
            for (int off = 16; off; off >>= 1) {
                const float ow = __shfl_xor_sync(kFull, bw, off); const long long os = __shfl_xor_sync(kFull, bs, off);
                const int oi = __shfl_xor_sync(kFull, bi, off);
                if (oi >= 0 && (bi < 0 || key_less(ow, os, bw, bs))) { bw = ow; bs = os; bi = oi; }
            }
            if (lane == 0) { s_head = bi; s_head_w = bw; s_tcount = 0; }
        }
        __syncthreads();
        const int head = s_head;
        PHASE(0);
        if (head < 0 || !(s_head_w < threshold)) break;          // strict <, src/clustering.cpp:388-389
        const unsigned a = E.a[head], b = E.b[head];
        __syncthreads();
        if (tid == 0) {
            const unsigned m = s_nm;
            if (m < log_cap) {                                    // debug line of :390-392
                mlog.a[m] = sv_label[a]; mlog.b[m] = sv_label[b]; mlog.w[m] = s_head_w;
                mlog.edges_left[m] = s_ealive; mlog.regions_left[m] = s_ralive;
            }
            E.stamp[head] = kDeadStamp; pk[head] = P::kDead;
            s_dirty[F3PS_OWNER(head)] = 1;
            s_lanes = (pos_data != nullptr && (float)R.n[a] + (float)R.n[b] < 16000000.0f) ? 1 : 0;
        }
        __syncthreads();
        // ---- B: fold (warp 0: covariance sums + eigen-solve, warp 1: colour mean + Lab)  ||  touched-edge scan (warps 2..31) ----
        if (warp == 0 && !s_lanes) {
            const unsigned long long steps = merge_fold_fallback(R, ep, a, b, run_start, run_end, order, vox_xyz, lane);
            if (lane == 0) s_fold += steps;
        } else if (warp == 0) {
            const float4 a0 = R.accu0[a], a1 = R.accu1[a], a2 = R.accu2[a];
            const float acc[9] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w, a2.x};
            float v = 0.0f;
#pragma unroll
            for (int k = 0; k < 9; ++k) if (lane == k) v = acc[k];
            float cnt = (float)R.n[a];
            const unsigned steps = fold_rope_lanes<false>(v, cnt, R, b, run_start, run_end, pos_data, s_stage, lane);   // voxels_ = a ++ b  (:408)
            const long long t_tail = clock64();
            float accu[9];
#pragma unroll
            for (int k = 0; k < 9; ++k) accu[k] = __shfl_sync(kFull, v, k);
            if (lane == 0) {
                const int n_new = R.n[a] + (int)steps;
                R.accu0[a] = make_float4(accu[0], accu[1], accu[2], accu[3]);
                R.accu1[a] = make_float4(accu[4], accu[5], accu[6], accu[7]);
                R.accu2[a] = make_float4(accu[8], 0, 0, 0);
                R.n[a] = n_new;
                const float fn = (float)n_new;
                const float cx = accu[6] / fn, cy = accu[7] / fn, cz = accu[8] / fn;             // computeCentroid (:411-413)
                float n[3]; float curv;
                if (n_new < 3) { n[0] = n[1] = n[2] = nanf(""); curv = n[0]; }
                else plane_from_accu(accu, n_new, n, curv);                                       // computePointNormal (:415-417)
                flip_and_normalize(cx, cy, cz, n);                                                // :418-420
                R.centroid[a] = make_float4(cx, cy, cz, 0.0f);
                R.normal[a] = make_float4(n[0], n[1], n[2], curv);
                s_fold += steps;
                pc[7] += (unsigned long long)(clock64() - t_tail);
            }
        } else if (warp == 1 && s_lanes) {
            const float4 m4 = R.mean[a];                          // cnt, r, g, b   (ColorUtilities::mean_color's running mean)
            float v = lane == 0 ? m4.y : (lane == 1 ? m4.z : m4.w);
            float cnt = m4.x;
            fold_rope_lanes<true>(v, cnt, R, b, run_start, run_end, pos_data, s_stage2, lane);
            const float mr = __shfl_sync(kFull, v, 0), mg = __shfl_sync(kFull, v, 1), mb = __shfl_sync(kFull, v, 2);
            if (lane == 0) {
                R.mean[a] = make_float4(cnt, mr, mg, mb);
                float cv[3]; colour_vector(ep, mr, mg, mb, cv);
                R.cvec[a] = make_float4(cv[0], cv[1], cv[2], 0.0f);
            }
        } else if (warp >= 2 || (warp == 1 && !s_lanes)) {
            constexpr unsigned kScan = kMergeThreads - 64;
            if (warp >= 2)
            for (unsigned base = tid - 64; base < nE; base += kScan * 8) {
                PK p[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) { const unsigned e = base + k * kScan; p[k] = e < nE ? __ldcg(pk + e) : P::kDead; }
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    if (p[k] == P::kDead) continue;
                    const unsigned e = base + k * kScan;
                    const unsigned ea = P::lo(p[k]), eb = P::hi(p[k]);
                    if ((int)e != head && (ea == a || eb == a || ea == b || eb == b)) {
                        const int slot = atomicAdd(&s_tcount, 1);
                        const unsigned x = (ea == a || ea == b) ? eb : ea;
                        if (slot < kMergeTcap) { sm_e[0][slot] = (int)e; sm_x[0][slot] = x; } else { scr.e[0][slot] = (int)e; scr.x[0][slot] = x; }
                    }
                }
            }
        }
        PHASE(1);                                                    // thread 0 folds: its own time
        __syncthreads();
        PHASE(5);                                                    // ... and what it then waits for the scan
        if (tid == 0) {                                              // the ropes: a ++ b; b is erased (:426-429)
            R.next_run[R.tail[a]] = R.head[b]; R.tail[a] = R.tail[b];
            R.n[b] = 0;
        }
        const int T = s_tcount;
        const bool big = T > kMergeTcap;
        if (tid == 0) pc[6] += (unsigned long long)T;
        if (big) {                                                   // rare: continue in the global scratch
            for (int i = tid; i < kMergeTcap; i += kMergeThreads) { scr.e[0][i] = sm_e[0][i]; scr.x[0][i] = sm_x[0][i]; }
            __syncthreads();
        }
        int* const s_e[2] = {big ? scr.e[0] : sm_e[0], big ? scr.e[1] : sm_e[1]};
        float* const s_w[2] = {big ? scr.w[0] : sm_w[0], big ? scr.w[1] : sm_w[1]};
        long long* const s_st[2] = {big ? scr.st[0] : sm_st[0], big ? scr.st[1] : sm_st[1]};
        unsigned* const s_x[2] = {big ? scr.x[0] : sm_x[0], big ? scr.x[1] : sm_x[1]};
        unsigned char* const s_class = big ? scr.cls : sm_cls;
        // ---- C: order the touched edges by their old key ---------------------------------
        if (!big) {
            for (int i = tid; i < T; i += kMergeThreads) {
                const int e = s_e[0][i];
                s_w[0][i] = E.w[e]; s_st[0][i] = E.stamp[e];
            }
            __syncthreads();
            for (int i = tid; i < T; i += kMergeThreads) {
                const float w = s_w[0][i]; const long long st = s_st[0][i];
                int r = 0;
                for (int j = 0; j < T; ++j) r += key_less(s_w[0][j], s_st[0][j], w, st) ? 1 : 0;
                s_e[1][r] = s_e[0][i]; s_w[1][r] = w; s_st[1][r] = st; s_x[1][r] = s_x[0][i];
            }
            __syncthreads();
        } else {
            // thousands of touched edges (a region with thousands of neighbours): bitonic sort of (old key, slot) records,
            // in shared memory up to 8192 records, else in the global buffer
            unsigned n2 = 2048; while (n2 < (unsigned)T) n2 <<= 1;
            MergeSortRec* buf = n2 <= (unsigned)kMergeSortSmem ? reinterpret_cast<MergeSortRec*>(dyn_smem) : scr.sortbuf;
            for (unsigned i = tid; i < n2; i += kMergeThreads) {
                MergeSortRec r;
                if (i < (unsigned)T) { const int e = s_e[0][i]; r.w = E.w[e]; r.st = E.stamp[e]; r.slot = i; }
                else { r.w = INF; r.st = kDeadStamp; r.slot = 0xffffffffu; }
                buf[i] = r;
            }
            __syncthreads();
            for (unsigned k = 2; k <= n2; k <<= 1) {
                for (unsigned j = k >> 1; j > 0; j >>= 1) {
                    for (unsigned i = tid; i < n2; i += kMergeThreads) {
                        const unsigned ixj = i ^ j;
                        if (ixj > i) {
                            const MergeSortRec ra = buf[i], rb = buf[ixj];
                            const bool up = (i & k) == 0;
                            if (key_less(rb.w, rb.st, ra.w, ra.st) == up) { buf[i] = rb; buf[ixj] = ra; }
                        }
                    }
                    __syncthreads();
                }
            }
            for (int r = tid; r < T; r += kMergeThreads) {
                const MergeSortRec q = buf[r];
                s_e[1][r] = s_e[0][q.slot]; s_w[1][r] = q.w; s_st[1][r] = q.st; s_x[1][r] = s_x[0][q.slot];
            }
            __syncthreads();
        }
        PHASE(2);
        // ---- D: dedupe (earlier survives), recompute, classify ---------------------------
        if (big) {                                                    // the earliest entry of every far end x survives
            for (int i = tid; i < T; i += kMergeThreads) atomicMin(&scr.mark[s_x[1][i]], (unsigned)i);
            __syncthreads();
        }
        for (int i = tid; i < T; i += kMergeThreads) {
            const unsigned x = s_x[1][i];
            bool dup = false;
            if (big) dup = scr.mark[x] != (unsigned)i;
            else for (int q = 0; q < i; ++q) dup = dup || (s_x[1][q] == x);
            if (dup) s_class[i] = C_DUP;
            else {
                const unsigned lo = min(a, x), hi = max(a, x);
                float rgb1[3], n1[3], c1[3], rgb2[3], n2[3], c2[3];
                region_inputs(R, (int)lo, rgb1, n1, c1); region_inputs(R, (int)hi, rgb2, n2, c2);
                float dc, dg;
                delta_cached(ep, rgb1, rgb2, n1, c1, n2, c2, dc, dg);
                float w_new = unify(ep, dc, dg);
                E.dc[s_e[1][i]] = dc;                              // the resident kernel memoises delta_c per edge: keep its copy current
                if (isnan(w_new)) { atomicAdd(&ctl->nan_weights, 1u); w_new = INF; }
                const float w_old = s_w[1][i];
                s_class[i] = (w_new == w_old) ? C_KEEP : (w_new > w_old ? C_FRONT : C_BACK);
                s_w[0][i] = w_new;                                 // slot 0 of the scratch is free again: new weights
            }
        }
        __syncthreads();
        PHASE(3);
        // ---- E: tie stamps (C.2) and write back -------------------------------------------
        if (!big) {
            // one entry per thread: ranks among the BACK / FRONT classes from ballots
            const int cls = tid < T ? (int)s_class[tid] : -1;
            const unsigned mb = __ballot_sync(kFull, cls == C_BACK), mf = __ballot_sync(kFull, cls == C_FRONT), md = __ballot_sync(kFull, cls == C_DUP);
            if (lane == 0) { s_wb[warp] = __popc(mb); s_wf[warp] = __popc(mf); s_wd[warp] = __popc(md); }
            __syncthreads();
            int nb = 0, nf = 0, nd = 0, rb = 0, rf = 0;
#pragma unroll
            for (int w = 0; w < 32; ++w) {
                const int wb = (int)s_wb[w], wf = (int)s_wf[w];
                nb += wb; nf += wf; nd += (int)s_wd[w];
                if (w < warp) { rb += wb; rf += wf; }
            }
            const unsigned lt = (1u << lane) - 1u;
            rb += __popc(mb & lt); rf += __popc(mf & lt);
            if (tid < T) {
                const int e = s_e[1][tid];
                if (cls == C_DUP) { E.stamp[e] = kDeadStamp; pk[e] = P::kDead; }
                else {
                    long long st = s_st[1][tid];
                    if (cls == C_BACK) st = s_counter + rb;
                    else if (cls == C_FRONT) st = -(s_counter + nb + (nf - 1 - rf));
                    const unsigned x = s_x[1][tid];
                    E.a[e] = min(a, x); E.b[e] = max(a, x); E.w[e] = s_w[0][tid]; E.stamp[e] = st;
                    pk[e] = P::pack(min(a, x), max(a, x));
                }
                s_dirty[F3PS_OWNER(e)] = 1;
            }
            __syncthreads();
            if (tid == 0) {
                s_counter += nb + nf;
                s_ealive -= 1 + nd; s_ralive -= 1; s_nm += 1;
                if ((unsigned)T > s_maxT) s_maxT = (unsigned)T;
            }
        } else {
            // ranks among the BACK / FRONT classes in old-key order: ballot scan, 1024 entries per round; the ranks are parked
            // in the (now free) slot-order arrays
            int* const rank_b = s_e[0]; unsigned* const rank_f = s_x[0];
            int nb = 0, nf = 0, nd = 0;
            for (int c0 = 0; c0 < T; c0 += kMergeThreads) {
                const int i = c0 + tid;
                const int cls = i < T ? (int)s_class[i] : -1;
                if (i < T) scr.mark[s_x[1][i]] = 0xffffffffu;             // marks back to "free" for the next merge
                const unsigned mb = __ballot_sync(kFull, cls == C_BACK), mf = __ballot_sync(kFull, cls == C_FRONT), md = __ballot_sync(kFull, cls == C_DUP);
                if (lane == 0) { s_wb[warp] = __popc(mb); s_wf[warp] = __popc(mf); s_wd[warp] = __popc(md); }
                __syncthreads();
                int rb = nb, rf = nf;
#pragma unroll
                for (int w = 0; w < 32; ++w) {
                    const int wb = (int)s_wb[w], wf = (int)s_wf[w];
                    if (w < warp) { rb += wb; rf += wf; }
                    nb += wb; nf += wf; nd += (int)s_wd[w];
                }
                const unsigned lt = (1u << lane) - 1u;
                if (i < T) { rank_b[i] = rb + __popc(mb & lt); rank_f[i] = (unsigned)(rf + __popc(mf & lt)); }
                __syncthreads();
            }
            for (int i = tid; i < T; i += kMergeThreads) {
                const int cls = s_class[i];
                const int e = s_e[1][i];
                if (cls == C_DUP) { E.stamp[e] = kDeadStamp; pk[e] = P::kDead; }
                else {
                    long long st = s_st[1][i];
                    if (cls == C_BACK) st = s_counter + rank_b[i];
                    else if (cls == C_FRONT) st = -(s_counter + nb + (nf - 1 - (int)rank_f[i]));
                    const unsigned x = s_x[1][i];
                    E.a[e] = min(a, x); E.b[e] = max(a, x); E.w[e] = s_w[0][i]; E.stamp[e] = st;
                    pk[e] = P::pack(min(a, x), max(a, x));
                }
                s_dirty[F3PS_OWNER(e)] = 1;
            }
            __syncthreads();
            if (tid == 0) {
                s_counter += nb + nf;
                s_ealive -= 1 + nd; s_ralive -= 1; s_nm += 1;
                if ((unsigned)T > s_maxT) s_maxT = (unsigned)T;
            }
        }
        __syncthreads();
        PHASE(4);
    }
    if (tid == 0) {
        for (int i = 0; i < 8; ++i) ctl->phase_cycles[i] = pc[i];
        ctl->n_merges = s_nm; ctl->edges_alive = s_ealive; ctl->regions_alive = s_ralive; ctl->counter = s_counter;
        ctl->fold_steps = s_fold; ctl->max_touched = s_maxT;
    }
}

} // namespace f3ps
