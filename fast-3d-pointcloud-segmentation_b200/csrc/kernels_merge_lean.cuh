// kernels_merge_lean.cuh -- K7, the resident kernel: Clustering::cluster / merge / contains
// (/root/reference/src/clustering.cpp:384-469, 497-506) replayed by ONE persistent CTA whose working set lives on the SM
// (SURVEY.md Appendix C for the replay rules).  Round 2 rewrite of the round-1 resident kernel: that one spent its time
// refetching instructions (8.9 k SASS instructions against a 32 KB instruction cache, 75 % hit rate) and ran CIEDE2000 on
// 128 of its 1024 threads.  This one keeps the per-merge code small and flat:
//
//   edges         shared memory: 64-bit order key (weight bits : biased tie stamp) + packed (a,b); worker warp w owns the blocks
//                 of 32 edges w, w + 29, ... and rescans them (independent loads) only after a merge re-weighted one of them
//   adjacency     per region a list of edge ids in an L2-resident pool (start / length / capacity in shared memory): the edges a
//                 merge touches are read from the two lists, never searched for; the survivors become a's new list
//   ropes / sizes shared memory (per region: head / tail / next run, run bounds, voxel count)
//   voxels        position-ordered float4 (x,y,z,rgba) in HBM/L2; a region of <= 256 voxels is fetched by the fold warps themselves
//                 (16-byte cp.async per lane, every run in flight at once); longer ones stream through a two-slot ring of 256
//                 voxels filled by the loader warp the same way (full/empty mbarriers, cp.async.mbarrier.arrive).  One bulk copy
//                 (TMA) per run, as in round 1, made the loader the bottleneck of the long folds: runs are ~15 voxels
//   touched edges ONE worker thread per touched edge (up to 928): duplicates through a per-region mark, CIEDE2000 in every
//                 thread that needs it (the round-1 kernel looped 128 threads over up to 600 edges), tie stamps through a hash
//
// Roles: warp 0 covariance / xyz sums + eigen-solve, warp 1 running colour mean + Lab, warp 2 loader, warps 3..31 workers.
// Barriers per merge: S1 (all: partial minima published), W1 (workers: touched list complete), WB1 / WB2 (workers, or one
// warp when <= 32 edges are touched), F (all: new geometry published), W4 (workers: new keys written).
//
// Two instantiations: tables in shared memory (S <= 4096, E <= 928 * 32, 12 E + 26 S + 40 KB within 227 KB: a VGA frame), or --
// BIG -- the per-edge / per-region tables in global memory with per-block minima in shared memory (S < 65535, 32-bit edge ids,
// E bounded by 16 bytes of shared memory per block of 32 edges: C4 / C5-size scenes).  Shared-memory variant: a merge whose two
// adjacency lists hold more than 928 entries is not started: every role stops in front of it, the state written back is that
// after n merges, and the host relaunches the BIG variant from that state with A.resume (f3ps.cu: merge_frames).  BIG variant:
// such a merge runs in lean_wide_merge (every worker thread loops over the entries, per-entry state in a global scratch); it
// stops only in front of a merge with more than 65,534 entries.  That stop, an exhausted adjacency pool or an exhausted stamp
// range makes the host replay the whole sequence again on merge_kernel (kernels_merge.cuh), from the initial state.
#pragma once
#include "kernels_merge.cuh"

namespace f3ps {

constexpr int kFastThreads = 1024;
constexpr int kLeanRoleWarps = 3;
constexpr int kFastOwners = kFastThreads - 32 * kLeanRoleWarps;     // 928 worker threads
constexpr int kLeanWorkerWarps = kFastOwners / 32;                  // 29
constexpr int kLeanMaxTouched = kFastOwners;
constexpr int kLeanHash = 1024;                      // tie-group table (distinct new weights of one merge), power of two
constexpr int kLeanHashShift = 22;                   // 32 - log2(kLeanHash)
constexpr int kLeanRing = 2, kLeanSlotVox = 256;     // (four slots measured no faster than two; 8 KB decide whether a VGA frame fits)
constexpr unsigned kDeadKey = 0xffffffffu;
constexpr unsigned long long kDeadKey64 = ~0ull;
constexpr unsigned kNil16 = 0xffffu;
constexpr unsigned kFastErrTouched = 4u;
constexpr unsigned kFastErrStamp = 8u;
constexpr unsigned kFastErrPool = 16u;
// BIG variant: a merge whose two adjacency lists hold more entries than there are worker threads (a floor or a wall of a dense scene
// has thousands of neighbours) keeps its per-entry state in a global scratch (L2) and every worker thread loops over the entries
// i, i + 928, ...  Entry indices travel in the 16-bit region marks, so the limit is 65,534 entries.
constexpr int kLeanWideMax = 65534;
constexpr unsigned kLeanWideSlots = 65536u;
constexpr unsigned kLeanWideHash = 1u << 17;         // tie-group table of a wide merge (distinct new weights), power of two
constexpr int kLeanWideHashShift = 15;               // 32 - log2(kLeanWideHash)
struct LeanWideScratch {
    unsigned long long *te_key, *nkey; unsigned *te_e, *res_w, *xs; float* dcs; unsigned* hs; unsigned short* partner; unsigned char *cls, *flags;
    unsigned *hkey, *hcnt;
    static constexpr size_t bytes = (size_t)kLeanWideSlots * (8 + 8 + 4 + 4 + 4 + 4 + 4 + 2 + 1 + 1) + (size_t)kLeanWideHash * 8;
    __host__ __device__ explicit LeanWideScratch(char* p) {
        te_key = (unsigned long long*)p; p += (size_t)kLeanWideSlots * 8; nkey = (unsigned long long*)p; p += (size_t)kLeanWideSlots * 8;
        xs = (unsigned*)p; p += (size_t)kLeanWideSlots * 4;
        te_e = (unsigned*)p; p += (size_t)kLeanWideSlots * 4; res_w = (unsigned*)p; p += (size_t)kLeanWideSlots * 4;
        dcs = (float*)p; p += (size_t)kLeanWideSlots * 4; hs = (unsigned*)p; p += (size_t)kLeanWideSlots * 4;
        partner = (unsigned short*)p; p += (size_t)kLeanWideSlots * 2;
        cls = (unsigned char*)p; p += kLeanWideSlots; flags = (unsigned char*)p; p += kLeanWideSlots;
        hkey = (unsigned*)p; p += (size_t)kLeanWideHash * 4; hcnt = (unsigned*)p;
    }
};

struct FastArgs {
    RegionArrays R; EdgeArrays E;
    const unsigned* n_edges_ptr; const unsigned* n_sv_ptr;
    EdgeParams ep; const float* lambda_dev; float threshold;
    const unsigned* run_start; const unsigned* run_end;
    const float4* pos_data;                  // voxel (x,y,z,rgba) by position of the label-ordered list
    const unsigned* sv_label;
    MergeLog mlog; unsigned log_cap;
    MergeCtl* ctl;
    unsigned short* adj_pool; unsigned pool_cap;   // adjacency lists (edge ids: 16 bits, BIG variant 32 bits), bump-allocated; capacity in entries
    unsigned* trace; unsigned trace_first;         // PROF only: clock() of 32 points of 256 merges starting at trace_first (f3ps_get_merge_trace)
    int resume;                              // continue a replay from the state in the edge / region arrays (counters in *ctl): the BIG variant after the shared-memory one stopped
    char* big; unsigned* big_cursor;         // BIG variant only: the per-edge / per-region tables (12 E_cap + 26 S_cap bytes) and the set-up scratch (4 S_cap) in global memory; LeanWideScratch sits at big_cursor + lean_cursor_bytes(S_cap)
    unsigned S_cap, E_cap;                   // table capacities the shared-memory layout was sized for (E_cap = E rounded up to whole blocks of 32 edges)
};

// shared-memory layout, shared by host (size) and device (pointers)
struct FastSmem {
    unsigned long long* key; unsigned* ab;
    float4* stage; unsigned long long* mbar;                        // full[kLeanRing], empty[kLeanRing]
    float4* priv;                                                   // one private stage per fold warp: regions of <= kLeanSlotVox voxels skip the loader
    unsigned short* partner; unsigned* res_w; unsigned char* cls; unsigned long long* te_key;
    unsigned *hkey, *hcnt;
    unsigned long long* wm_key; unsigned *wm_e, *wm_ab;
    float* newgeo; int* misc; float* inv; unsigned* bdirty;
    unsigned* rs; unsigned short* rlen; int* n;
    unsigned short *head, *tail, *next, *mark;
    unsigned* adj_start; unsigned short *adj_len, *adj_cap;
    size_t bytes;
    // Fixed-size tables first (compile-time offsets), then the two per-edge tables, then the per-region ones: every pointer is
    // base + constant (+ k * E_cap) (+ k * S) with S a multiple of 8 and E_cap a multiple of 32, so no alignment rounding depends
    // on a run-time value.  (ncu, round 2: the generic bump allocator this replaces cost 8 % of the kernel's instructions --
    // the 30 pointers do not fit the 64 registers and were re-derived through its dependent additions all over the merge loop.)
    // BIG variant (graphs that do not fit an SM: S up to 65,534, E up to 65,504): the per-edge and per-region tables live in global
    // memory (`big`, L2-resident) and shared memory keeps, per block of 32 edges, the block's minimum key with its edge and end
    // points (bm_*) and a dirty bit -- a re-weighted edge costs its block one coalesced 256-byte reload, never a scan of the map.
    unsigned long long* bm_key; unsigned *bm_e, *bm_ab, *blkdirty;
    __host__ __device__ FastSmem(char* base, unsigned S, unsigned E_cap, char* big = nullptr) {
        size_t o = 0;
        auto take = [&](size_t b) { char* p = base + o; o += (b + 15) & ~(size_t)15; return p; };
        mbar = (unsigned long long*)take(2 * kLeanRing * 8);
        stage = (float4*)take((size_t)kLeanRing * kLeanSlotVox * 16);
        priv = (float4*)take((size_t)2 * kLeanSlotVox * 16);     // directly behind the ring: the set-up's scratch (4 bytes per region, S <= 4096) spans both
        te_key = (unsigned long long*)take(kLeanMaxTouched * 8);
        partner = (unsigned short*)take(kLeanMaxTouched * 2);
        res_w = (unsigned*)take(kLeanMaxTouched * 4); cls = (unsigned char*)take(kLeanMaxTouched);
        hkey = (unsigned*)take(kLeanHash * 4); hcnt = (unsigned*)take(kLeanHash * 4);
        wm_key = (unsigned long long*)take(32 * 8); wm_e = (unsigned*)take(32 * 4); wm_ab = (unsigned*)take(32 * 4);
        newgeo = (float*)take(16 * 4); misc = (int*)take(16 * 4); inv = (float*)take(64 * 4); bdirty = (unsigned*)take(32 * 4);
        char* eb = base + o;                                      // o is a compile-time constant up to here
        bm_key = nullptr; bm_e = bm_ab = blkdirty = nullptr;
        if (big) {
            const size_t nblk = E_cap / 32u;
            bm_key = (unsigned long long*)eb; bm_e = (unsigned*)(eb + nblk * 8); bm_ab = (unsigned*)(eb + nblk * 12);
            blkdirty = (unsigned*)(eb + nblk * 16);
            o += nblk * 16 + ((nblk + 31) / 32) * 4;
            eb = big;
        }
        key = (unsigned long long*)eb; ab = (unsigned*)(eb + (size_t)E_cap * 8);
        char* const sb = eb + (size_t)E_cap * 12;
        rs = (unsigned*)sb; n = (int*)(sb + (size_t)S * 4); adj_start = (unsigned*)(sb + (size_t)S * 8);
        rlen = (unsigned short*)(sb + (size_t)S * 12); head = (unsigned short*)(sb + (size_t)S * 14); tail = (unsigned short*)(sb + (size_t)S * 16);
        next = (unsigned short*)(sb + (size_t)S * 18); mark = (unsigned short*)(sb + (size_t)S * 20);
        adj_len = (unsigned short*)(sb + (size_t)S * 22); adj_cap = (unsigned short*)(sb + (size_t)S * 24);
        bytes = big ? o : o + (size_t)E_cap * 12 + (size_t)S * 26;
    }
    static __host__ __device__ size_t big_bytes(unsigned S, unsigned E_cap) { return (size_t)E_cap * 12 + (size_t)S * 26 + 256; }
};
__host__ __device__ inline size_t lean_cursor_bytes(unsigned S_cap) { return ((size_t)S_cap * 4 + 255) & ~(size_t)255; }
enum { FM_NLIVE = 0, FM_EALIVE, FM_RALIVE, FM_COUNTER, FM_ND, FM_NANW, FM_ERROR, FM_MAXT, FM_SUMT, FM_MISS, FM_EVALS, FM_NMERGES, FM_POOL };

// ---- PTX helpers: mbarrier, cp.async, named barriers ------------------------
__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned mbar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_local(unsigned mbar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mbar) : "memory"); }
__device__ __forceinline__ void mbar_wait(unsigned mbar, unsigned parity) {
    unsigned ok;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(mbar), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void cp_async16(unsigned dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// A region of at most kLeanSlotVox voxels: the fold warp copies its runs itself (one 16-byte cp.async per lane and voxel,
// every run in flight at once) -- one L2 round trip instead of the loader hand-over plus a bulk copy per run.
__device__ __forceinline__ void lean_fetch_small(const unsigned short* head, const unsigned short* next, const unsigned* rs, const unsigned short* rlen,
                                                 const float4* __restrict__ pos_data, unsigned b, int nb, float4* dst, int lane) {
    unsigned run = head[b]; int filled = 0;
    while (filled < nb && run != kNil16) {
        const unsigned r0 = rs[run]; const int len = (int)rlen[run];
        for (int j = lane; j < len; j += 32) cp_async16(smem_addr(dst + filled + j), pos_data + r0 + j);
        filled += len; run = next[run];
    }
    cp_async_wait_all();
    __syncwarp();
}
__device__ __forceinline__ void named_bar(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// OpenCV's LUT interpolation spread over 8 lanes (one lattice corner each); result valid in every lane of the warp
__device__ __forceinline__ void rgb2lab_lanes(const short* __restrict__ lut, float r255, float g255, float b255, int lane, float lab[3]) {
    const float in[3] = {r255, g255, b255};
    int t[3], f[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float v = in[k] / 255;
        v = fminf(fmaxf(v, 0.0f), 1.0f);
        const int c = (int)rintf(v * 16384.0f);
        t[k] = c >> 9; f[k] = (c >> 5) & 15;
    }
    int out[3] = {0, 0, 0};
    if (lane < 8) {
        const int dr = lane >> 2, dg = (lane >> 1) & 1, db = lane & 1;
        const int w = (dr ? f[0] : 16 - f[0]) * (dg ? f[1] : 16 - f[1]) * (db ? f[2] : 16 - f[2]);
        const int ir = min(t[0] + dr, 32), ig = min(t[1] + dg, 32), ib = min(t[2] + db, 32);
        const short* e = lut + ((ir * 33 + ig) * 33 + ib) * 3;
        out[0] = w * (int)e[0]; out[1] = w * (int)e[1]; out[2] = w * (int)e[2];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        int v = out[k];
        v += __shfl_xor_sync(kFull, v, 4); v += __shfl_xor_sync(kFull, v, 2); v += __shfl_xor_sync(kFull, v, 1);
        out[k] = (__shfl_sync(kFull, v, 0) + 2048) >> 12;
    }
    lab[0] = ((float)out[0] / 16384.0f) * 100.0f;
    lab[1] = ((float)out[1] / 16384.0f) * 256.0f - 128.0f;
    lab[2] = ((float)out[2] / 16384.0f) * 256.0f - 128.0f;
}

// delta_c of Clustering::delta_c_g (src/clustering.cpp:113-122) on two colour vectors, first argument = smaller label.
// One copy of the FP64 code in the kernel (the instruction cache, not the FP64 pipe, bounds a replicated version).
__device__ __noinline__ float colour_delta(int color_mode, float4 lo, float4 hi) {
    const float c1[3] = {lo.x, lo.y, lo.z}, c2[3] = {hi.x, hi.y, hi.z};
    float dc;
    if (color_mode == 0) { dc = lab_ciede00(c1, c2); dc /= F3PS_LAB_RANGE; }
    else { dc = rgb_eucl(c1, c2); dc /= F3PS_RGB_RANGE; }
    return dc;
}

// delta_g of Clustering::delta_c_g (src/clustering.cpp:126-138), first argument = smaller label: normals_diff (:79-96) and
// is_convex (:53-67) share the unit centroid difference and the two projections (the same float expressions in both).
__device__ __forceinline__ float geom_delta(int geom_mode, float4 n1, float4 c1, float4 n2, float4 c2) {
    float C0 = c1.x - c2.x, C1 = c1.y - c2.y, C2 = c1.z - c2.z;
    const float nrm = sqrtf(sum3(C0 * C0, C1 * C1, C2 * C2));
    C0 /= nrm; C1 /= nrm; C2 /= nrm;
    const float x0 = n1.y * n2.z - n1.z * n2.y, x1 = n1.z * n2.x - n1.x * n2.z, x2 = n1.x * n2.y - n1.y * n2.x;
    const float N1xN2 = sqrtf(sum3(x0 * x0, x1 * x1, x2 * x2));
    const float cos1 = sum3(n1.x * C0, n1.y * C1, n1.z * C2), cos2 = sum3(n2.x * C0, n2.y * C1, n2.z * C2);
    float dg = (N1xN2 + fabsf(cos1) + fabsf(cos2)) / 3;
    if (geom_mode == 1 && cos1 >= cos2) dg *= 0.5f;
    return dg;
}

// computeCentroid + computePointNormal + flipNormalTowardsViewpoint of Clustering::merge (src/clustering.cpp:411-424) on the nine
// raw sums held one per lane (lane k < 9: accu[k] of plane_from_accu), spread over the lanes of one warp: every group of
// independent IEEE divisions (9 by n, 6 by the scale, 3 + 3 normalisations) and the three cross products run once, side by
// side, instead of back to back in one thread.  Same float expressions in the same association order as plane_from_accu /
// eigen33_smallest / flip_and_normalize (kernels_vccs.cuh): bit-identical results, valid in every lane.
__device__ __forceinline__ void plane_from_accu_warp(float acc, int nn, int lane, int pi, int qi, float cen[3], float nv[3], float& curv) {
    const float fn = (float)nn;
    const float am = acc / fn;                                                                // accu[k] / n  (k = lane)
    cen[0] = __shfl_sync(kFull, am, 6); cen[1] = __shfl_sync(kFull, am, 7); cen[2] = __shfl_sync(kFull, am, 8);
    if (nn < 3) { nv[0] = nv[1] = nv[2] = nanf(""); curv = nv[0]; }
    else {
        const float ap = __shfl_sync(kFull, am, 6 + pi), aq = __shfl_sync(kFull, am, 6 + qi);
        const float cov = am - ap * aq;                                                       // lanes 0..5: xx xy xz yy yz zz
        float sc = lane < 6 ? fabsf(cov) : 0.0f;
        sc = fmaxf(sc, __shfl_xor_sync(kFull, sc, 4)); sc = fmaxf(sc, __shfl_xor_sync(kFull, sc, 2)); sc = fmaxf(sc, __shfl_xor_sync(kFull, sc, 1));
        sc = __shfl_sync(kFull, sc, 0);
        if (sc <= FLT_MIN) sc = 1.0f;
        const float smk = cov / sc;
        const float m00 = __shfl_sync(kFull, smk, 0), m01 = __shfl_sync(kFull, smk, 1), m02 = __shfl_sync(kFull, smk, 2);
        const float m11 = __shfl_sync(kFull, smk, 3), m12 = __shfl_sync(kFull, smk, 4), m22 = __shfl_sync(kFull, smk, 5);
        const float mm[9] = {m00, m01, m02, m01, m11, m12, m02, m12, m22};
        float roots[3];
        compute_roots(mm, roots);
        const float ev = roots[0] * sc;
        const float d00 = m00 - roots[0], d11 = m11 - roots[0], d22 = m22 - roots[0];
        // lane 0: row0 x row1, lane 1: row0 x row2, lane 2: row1 x row2
        const bool second = lane == 2, first = lane == 0;
        const float a0 = second ? m01 : d00, a1 = second ? d11 : m01, a2 = second ? m12 : m02;
        const float b0 = first ? m01 : m02, b1 = first ? d11 : m12, b2 = first ? m12 : d22;
        const float v0 = a1 * b2 - a2 * b1, v1 = a2 * b0 - a0 * b2, v2 = a0 * b1 - a1 * b0;
        const float l = sum3(v0 * v0, v1 * v1, v2 * v2);
        const float l1 = __shfl_sync(kFull, l, 0), l2 = __shfl_sync(kFull, l, 1), l3 = __shfl_sync(kFull, l, 2);
        const int which = (l1 >= l2 && l1 >= l3) ? 0 : ((l2 >= l1 && l2 >= l3) ? 1 : 2);
        const float s = sqrtf(which == 0 ? l1 : (which == 1 ? l2 : l3));
        const float w0 = __shfl_sync(kFull, v0, which), w1 = __shfl_sync(kFull, v1, which), w2 = __shfl_sync(kFull, v2, which);
        const float comp = (lane == 0 ? w0 : (lane == 1 ? w1 : w2)) / s;                       // lanes 0..2: one component each
        nv[0] = __shfl_sync(kFull, comp, 0); nv[1] = __shfl_sync(kFull, comp, 1); nv[2] = __shfl_sync(kFull, comp, 2);
        const float c0 = __shfl_sync(kFull, cov, 0), c3 = __shfl_sync(kFull, cov, 3), c5 = __shfl_sync(kFull, cov, 5);
        const float eig_sum = c0 + c3 + c5;
        curv = (eig_sum != 0) ? fabsf(ev / eig_sum) : 0.0f;
    }
    // flipNormalTowardsViewpoint(p, 0,0,0, n) ; n[3]=0 ; normalize()
    const float cos_theta = sum4((0.0f - cen[0]) * nv[0], (0.0f - cen[1]) * nv[1], (0.0f - cen[2]) * nv[2], 0.0f);
    if (cos_theta < 0) { nv[0] *= -1; nv[1] *= -1; nv[2] *= -1; }
    const float z = sum4(nv[0] * nv[0], nv[1] * nv[1], nv[2] * nv[2], 0.0f);
    if (z > 0.0f) {
        const float sz = sqrtf(z);
        const float comp = (lane == 0 ? nv[0] : (lane == 1 ? nv[1] : nv[2])) / sz;
        nv[0] = __shfl_sync(kFull, comp, 0); nv[1] = __shfl_sync(kFull, comp, 1); nv[2] = __shfl_sync(kFull, comp, 2);
    }
}

struct FastHead { unsigned hi, lo, e, ab; };
// every warp derives the head of the weight map from the worker warps' partial minima (after S1)
__device__ __forceinline__ FastHead lean_head(const FastSmem& sm, int lane) {
    FastHead h;
    const unsigned long long k = lane < kLeanWorkerWarps ? sm.wm_key[lane] : kDeadKey64;
    const unsigned hi = (unsigned)(k >> 32), lo = (unsigned)k;
    h.hi = __reduce_min_sync(kFull, hi);
    h.lo = __reduce_min_sync(kFull, hi == h.hi ? lo : kDeadKey);
    const int win = __ffs(__ballot_sync(kFull, hi == h.hi && lo == h.lo)) - 1;
    h.e = sm.wm_e[win]; h.ab = sm.wm_ab[win];
    return h;
}

// BIG variant, an edge of block e / 32 goes from key `okey` to `nkey` (dead = removed): a key below the block's cached minimum
// becomes the minimum by atomicMin (its edge id / end points are written after the next worker barrier by the thread whose key
// won); only when the block's minimum edge itself moved up or died is the block reloaded (dirty bit, phase A).
__device__ __forceinline__ void lean_block_min_update(const FastSmem& sm, unsigned e, unsigned long long okey, unsigned long long nkey) {
    const unsigned blk = e >> 5;
    if (sm.bm_e[blk] == e && nkey > okey) atomicOr(&sm.blkdirty[blk >> 5], 1u << (blk & 31u));
    else if (nkey != kDeadKey64) atomicMin(&sm.bm_key[blk], nkey);
}
enum { FC_KEEP = 0, FC_FRONT = 1, FC_BACK = 2, FC_DUP = 3 };
enum { BAR_W1 = 1, BAR_WB = 2, BAR_F = 3, BAR_W4 = 4, BAR_G = 5, BAR_FN = 6, BAR_GN = 7 };
// A merge whose two adjacency lists hold <= 32 entries is NARROW: one worker warp handles it, the other 28 sleep until W4, and
// the G / F barriers shrink to the warps involved (G: mean warp + worker warp 0; F: the three role warps + worker warp 0).
template <bool BIG, int NT>
__device__ __forceinline__ bool lean_too_wide(const FastSmem& sm, unsigned a, unsigned b) {
    return (unsigned)sm.adj_len[a] + (unsigned)sm.adj_len[b] > (unsigned)(BIG ? kLeanWideMax : NT - 32 * kLeanRoleWarps);
}
__device__ __forceinline__ bool lean_wide(const FastSmem& sm, unsigned a, unsigned b) { return (unsigned)sm.adj_len[a] + (unsigned)sm.adj_len[b] > 32u; }
__device__ __forceinline__ void bar_arrive(int id, int nthreads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// BIG variant, a merge with more adjacency entries than worker threads (T > 928): the same steps as the one-entry-per-thread
// code in merge_lean_body -- C (entries, duplicates through the region marks), colour deltas against the guess, D (geometry,
// weight, class, tie groups, a's new list), E (tie stamps, new keys) -- with every worker thread looping over the entries
// i, i + 928, ... and the per-entry state parked in LeanWideScratch between the barriers.  Same barrier protocol as a wide
// merge of the main loop (WB1, G, F, WB2; the caller arrives at W4).  Only the L2 variant instantiates it (a cold branch of its worker loop;
// inlined: as a separate function the call pinned the caller's table pointers to the stack).
template <bool PROF>
__device__ __forceinline__ void lean_wide_merge(const FastArgs& A, float lambda, unsigned head_e, unsigned a, unsigned b, int counter, unsigned pool_top, int wtid) {
    extern __shared__ __align__(128) char smem_raw[];
    const FastSmem sm(smem_raw, A.S_cap, A.E_cap, A.big);          // (rebuilt here: a reference would pin the caller's copy to its stack)
    EdgeParams ep = A.ep; ep.lambda = lambda;
    const int lane = wtid & 31;
    const RegionArrays& R = A.R;
    unsigned* const pool = reinterpret_cast<unsigned*>(A.adj_pool);
    const LeanWideScratch ws(reinterpret_cast<char*>(A.big_cursor) + lean_cursor_bytes(A.S_cap));
    const int* const newgeo_i = reinterpret_cast<const int*>(sm.newgeo);
    const unsigned la = sm.adj_len[a], lb = sm.adj_len[b], sa = sm.adj_start[a], sb = sm.adj_start[b];
    const unsigned ca = sm.adj_cap[a], cb = sm.adj_cap[b];
    const unsigned T = la + lb;
    unsigned t_prev = PROF ? (unsigned)clock() : 0u;
#define WIDE_PROF(k) do { if (PROF && wtid == 0) { const unsigned t_now = (unsigned)clock(); A.ctl->phase_cycles[20 + (k)] += t_now - t_prev; t_prev = t_now; } } while (0)
    // ---- C: entries, duplicates (a,x)/(b,x) through the region marks ----
    for (unsigned i = (unsigned)wtid; i < T; i += (unsigned)kFastOwners) {
        const unsigned e = __ldcg(pool + (i < la ? sa + i : sb + (i - la)));
        const unsigned eab = sm.ab[e];
        const bool mine = e != head_e && eab != kDeadKey;                                  // lists keep removed edges until they are rewritten
        ws.te_e[i] = mine ? e : kDeadKey;
        if (mine) {
            ws.te_key[i] = sm.key[e];
            const unsigned ea = eab >> 16, eb = eab & 0xffffu;
            const unsigned x = (ea == a || ea == b) ? eb : ea;
            ws.xs[i] = x | ((ea == a || eb == a) ? 0x10000u : 0u);                          // far end + "this edge hangs on a": the later phases do not go back to the edge table
            const unsigned short old = atomicCAS(&sm.mark[x], (unsigned short)kNil16, (unsigned short)i);
            if (old != (unsigned short)kNil16) { ws.partner[i] = old; ws.partner[old] = (unsigned short)i; }
        }
    }
    named_bar(BAR_WB, kFastOwners);                                                        // WB1
    named_bar(BAR_G, 32 + kFastOwners);                                                    // G: the guess of a's new colour vector
    WIDE_PROF(0);
    const float4 guess = make_float4(sm.newgeo[10], sm.newgeo[11], sm.newgeo[12], 0.0f);
    for (unsigned i = (unsigned)wtid; i < T; i += (unsigned)kFastOwners) {
        const unsigned e = __ldcg(ws.te_e + i);
        const unsigned xw = __ldcg(ws.xs + i);
        if (e == kDeadKey) continue;
        const bool side_a = (xw & 0x10000u) != 0u;
        const unsigned x = xw & 0xffffu;
        const unsigned long long okey = __ldcg(ws.te_key + i);
        const unsigned q = __ldcg(ws.partner + i);
        const bool dup = q != kNil16 && __ldcg(ws.te_key + q) < okey;                       // the earlier of (a,x), (b,x) survives
        sm.mark[x] = (unsigned short)kNil16; ws.partner[i] = (unsigned short)kNil16;
        const bool live = !dup;
        float dc = __ldcg(A.E.dc + e);
        const float4 xcv = __ldcg(R.cvec + x), ocv = __ldcg(R.cvec + (side_a ? a : b));
        const bool same_cv = __float_as_uint(ocv.x) == __float_as_uint(guess.x) && __float_as_uint(ocv.y) == __float_as_uint(guess.y) &&
                             __float_as_uint(ocv.z) == __float_as_uint(guess.z);
        const bool reuse = same_cv && (side_a || ((b < x) == (a < x)));
        const bool need = live && !reuse;
        if (need) { const bool af = a < x; dc = colour_delta(ep.color_mode, af ? guess : xcv, af ? xcv : guess); }
        ws.dcs[i] = dc; ws.flags[i] = (unsigned char)(live ? 1 : 0);
    }
    named_bar(BAR_F, kFastThreads);                                                        // F: region a's new colour vector / centroid / normal
    WIDE_PROF(1);
    // ---- D: colour delta after a wrong guess, geometry delta, weight, class, tie groups, a's new list ----
    const bool fresh = ca < T && cb < T;
    const unsigned ncap = fresh ? min(2u * T, 65535u) : (ca >= T ? ca : cb);
    const unsigned dst = ca >= T ? sa : (cb >= T ? sb : pool_top);
    const bool pool_ok = !fresh || pool_top + ncap <= A.pool_cap;
    const bool hit = newgeo_i[9] != 0;
    const float4 acv = make_float4(sm.newgeo[0], sm.newgeo[1], sm.newgeo[2], 0.0f);
    const float4 ace = make_float4(sm.newgeo[3], sm.newgeo[4], sm.newgeo[5], 0.0f), anr = make_float4(sm.newgeo[6], sm.newgeo[7], sm.newgeo[8], 0.0f);
    for (unsigned base = 0; base < T; base += (unsigned)kFastOwners) {                      // (uniform trip count: ballots inside)
        const unsigned i = base + (unsigned)wtid;
        const unsigned e = i < T ? __ldcg(ws.te_e + i) : kDeadKey;
        bool live = false;
        if (e != kDeadKey) {
            live = __ldcg(ws.flags + i) != 0;
            unsigned wbits = kDeadKey, hs = kDeadKey; int cls = FC_DUP;
            if (live) {
                const unsigned x = __ldcg(ws.xs + i) & 0xffffu;
                const bool a_first = a < x;
                float dc = __ldcg(ws.dcs + i);
                if (!hit) { const float4 xcv = __ldcg(R.cvec + x); dc = colour_delta(ep.color_mode, a_first ? acv : xcv, a_first ? xcv : acv); }   // wrong guess (rare)
                const float4 c4 = __ldcg(R.centroid + x), n4 = __ldcg(R.normal + x);
                const float dg = geom_delta(ep.geom_mode, a_first ? anr : n4, a_first ? ace : c4, a_first ? n4 : anr, a_first ? c4 : ace);
                float w_new = unify(ep, dc, dg);
                if (isnan(w_new)) { atomicAdd(&sm.misc[FM_NANW], 1); w_new = __int_as_float(0x7f800000); }
                wbits = __float_as_uint(w_new);
                const unsigned old_hi = (unsigned)(__ldcg(ws.te_key + i) >> 32);
                cls = wbits == old_hi ? FC_KEEP : (wbits > old_hi ? FC_FRONT : FC_BACK);
                if (cls != FC_KEEP) {                                                      // tie groups: same new weight, same side
                    const unsigned hk = wbits | (cls == FC_FRONT ? 0x80000000u : 0u);
                    unsigned h = (hk * 2654435761u) >> kLeanWideHashShift;
                    while (true) {
                        const unsigned prev = atomicCAS(&ws.hkey[h], kDeadKey, hk);
                        if (prev == hk) ws.hcnt[h] = 1u;                                   // a second entry with this weight and side: a tie group (rare)
                        if (prev == kDeadKey || prev == hk) break;
                        h = (h + 1) & (kLeanWideHash - 1);
                    }
                    hs = h;
                }
                A.E.dc[e] = dc;
            } else atomicAdd(&sm.misc[FM_ND], 1);
            ws.res_w[i] = wbits; ws.cls[i] = (unsigned char)cls; ws.hs[i] = hs;
        } else if (i < T) { ws.res_w[i] = kDeadKey; ws.cls[i] = (unsigned char)FC_DUP; ws.hs[i] = kDeadKey; }   // a removed edge's entry
        const unsigned lm = __ballot_sync(kFull, live);                                     // survivors take consecutive places in a's new list
        const int leader = __ffs(lm) - 1;
        int at = 0;
        if (lm && lane == leader) at = atomicAdd(&sm.misc[FM_NLIVE], __popc(lm));
        at = __shfl_sync(kFull, at, leader < 0 ? 0 : leader);
        if (live && pool_ok) pool[dst + (unsigned)at + (unsigned)__popc(lm & ((1u << lane) - 1u))] = e;
    }
    named_bar(BAR_WB, kFastOwners);                                                        // WB2
    WIDE_PROF(2);
    // ---- E: tie stamps, new keys ----
    for (unsigned base = 0; base < T; base += (unsigned)kFastOwners) {                      // (uniform trip count: the ranks are warp-wide scans)
        const unsigned i = base + (unsigned)wtid;
        const unsigned e = i < T ? __ldcg(ws.te_e + i) : kDeadKey;
        const bool mine = e != kDeadKey;
        bool live = false; unsigned long long okey = kDeadKey64; unsigned wbits = kDeadKey, hs = kDeadKey, gsz = 0; int cls = FC_DUP;
        if (mine) {
            live = __ldcg(ws.flags + i) != 0; okey = __ldcg(ws.te_key + i);
            wbits = __ldcg(ws.res_w + i); hs = __ldcg(ws.hs + i); cls = (int)__ldcg(ws.cls + i);
            if (hs != kDeadKey) gsz = 1u + __ldcg(ws.hcnt + hs);                            // 2 = "tied" (the group's size comes out of the rank scan)
        }
        // new arrivals keep their old relative order inside a tie group: rank = entries of the group (same tie slot) with a smaller
        // old key, counted by the whole warp for one tied lane after the other
        unsigned rank = 0;
        unsigned tied = __ballot_sync(kFull, gsz > 1u);
        while (tied) {
            const int src = __ffs(tied) - 1; tied &= tied - 1u;
            const unsigned s_hs = __shfl_sync(kFull, hs, src);
            const unsigned long long s_key = __shfl_sync(kFull, okey, src);
            unsigned cnt = 0, grp = 0;
#pragma unroll 8
            for (unsigned q = (unsigned)lane; q < T; q += 32u)
                if (__ldcg(ws.hs + q) == s_hs) { ++grp; if (__ldcg(ws.te_key + q) < s_key) ++cnt; }
            cnt = __reduce_add_sync(kFull, cnt); grp = __reduce_add_sync(kFull, grp);
            if (lane == src) { rank = cnt; gsz = grp; }
        }
        if (!mine) continue;
        unsigned lo = (unsigned)okey;
        if (hs != kDeadKey) {
            const int st = cls == FC_BACK ? counter + (int)rank : -(counter + (int)(gsz - 1 - rank));
            lo = (unsigned)st ^ 0x80000000u;
        }
        unsigned nab = kDeadKey;
        if (live) { const unsigned x = __ldcg(ws.xs + i) & 0xffffu; nab = a < x ? (a << 16) | x : (x << 16) | a; }
        const unsigned long long nkey = live ? ((unsigned long long)wbits << 32) | lo : kDeadKey64;
        ws.nkey[i] = nkey;
        sm.key[e] = nkey;
        sm.ab[e] = nab;
        sm.bdirty[(e >> 5) % kLeanWorkerWarps] = 1u;
        lean_block_min_update(sm, e, okey, nkey);
    }
    if (wtid == 0) {
        if (counter > 0x7f000000 - (int)T) sm.misc[FM_ERROR] = (int)kFastErrStamp;
        if (!pool_ok) sm.misc[FM_ERROR] = (int)kFastErrPool;
        else if (fresh) sm.misc[FM_POOL] = (int)(pool_top + ncap);
        sm.adj_start[a] = dst;
        sm.adj_len[a] = (unsigned short)sm.misc[FM_NLIVE]; sm.adj_cap[a] = (unsigned short)ncap; sm.adj_len[b] = 0; sm.adj_cap[b] = 0;
        sm.misc[FM_NLIVE] = 0;
        sm.misc[FM_COUNTER] = counter + (int)T;
        sm.misc[FM_EALIVE] -= 1 + sm.misc[FM_ND]; sm.misc[FM_ND] = 0; sm.misc[FM_RALIVE] -= 1;
        if ((int)T > sm.misc[FM_MAXT]) sm.misc[FM_MAXT] = (int)T;
        sm.misc[FM_SUMT] += (int)T; sm.misc[FM_MISS] += newgeo_i[9] ? 0 : 1;
    }
    named_bar(BAR_WB, kFastOwners);                                                        // every rank scan is done with the tie table; every atomicMin has landed
    for (unsigned i = (unsigned)wtid; i < T; i += (unsigned)kFastOwners) {
        const unsigned hs = __ldcg(ws.hs + i);
        if (hs != kDeadKey) { ws.hkey[hs] = kDeadKey; ws.hcnt[hs] = 0u; }
        const unsigned e = __ldcg(ws.te_e + i);
        if (e != kDeadKey && __ldcg(ws.flags + i) != 0) {                                   // the new block minima's edge / end points
            if (sm.bm_key[e >> 5] == __ldcg(ws.nkey + i)) {
                const unsigned x = __ldcg(ws.xs + i) & 0xffffu;
                sm.bm_e[e >> 5] = e; sm.bm_ab[e >> 5] = a < x ? (a << 16) | x : (x << 16) | a;
            }
        }
    }
    WIDE_PROF(3);
#undef WIDE_PROF
}

#define LPROF_DECL unsigned pc[8] = {0, 0, 0, 0, 0, 0, 0, 0}; unsigned t_prev = PROF ? (unsigned)clock() : 0u
#define LPROF(cond, i) do { if (PROF && (cond)) { const unsigned t_now = (unsigned)clock(); pc[i] += t_now - t_prev; t_prev = t_now; } } while (0)
#define LTRACE(cond, slot, val) do { if (PROF && (cond) && A.trace && (nm - A.trace_first) < 256u) A.trace[(nm - A.trace_first) * 32u + (slot)] = (val); } while (0)
#define LPROF_STORE(cond, base, n) do { if (PROF && (cond)) for (int i_ = 0; i_ < (n); ++i_) A.ctl->phase_cycles[(base) + i_] = pc[i_]; } while (0)

// NT = threads of the CTA: 1024 (29 worker warps, merges of up to 928 adjacency entries: what a grid of many frames runs, and the L2
// variant) or 768 (21 worker warps, 672 entries, 80 registers per thread instead of 64: a third of the spills and smaller
// barriers -- a VGA frame alone replays 11 % faster on it; a frame with a wider merge continues on the L2 variant, merge path 6).
template <bool PROF, bool BIG = false, int NT = 1024>
__device__ __forceinline__ void merge_lean_body(const FastArgs& A) {
    static_assert(!BIG || NT == 1024, "the L2 variant (lean_wide_merge) is written for 1024 threads");
    constexpr int kFastThreads = NT;                                    // (these shadow the namespace-scope constants of the 1024-thread layout)
    constexpr int kFastOwners = NT - 32 * kLeanRoleWarps;
    constexpr int kLeanWorkerWarps = kFastOwners / 32;
    constexpr int kLeanMaxTouched = kFastOwners;
    extern __shared__ __align__(128) char smem_raw[];
    const FastSmem sm(smem_raw, A.S_cap, A.E_cap, BIG ? A.big : nullptr);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned nE = *A.n_edges_ptr, S = *A.n_sv_ptr;
    const unsigned nm_first = A.resume ? A.ctl->n_merges : 0u;
    const RegionArrays R = A.R;
    const unsigned mbar_full = smem_addr(sm.mbar), mbar_empty = mbar_full + 8u * kLeanRing;
    int* const newgeo_i = reinterpret_cast<int*>(sm.newgeo);
    using PoolT = typename std::conditional<BIG, unsigned, unsigned short>::type;          // edge ids of the adjacency lists
    PoolT* const adj_pool = reinterpret_cast<PoolT*>(A.adj_pool);

    // ---- set-up: ropes, edges, adjacency lists -> shared memory / the pool ------------------------------------------------
    const unsigned nblk = A.E_cap / 32u;                                       // blocks of 32 edges; warp w owns w, w + 29, ...
    const unsigned nbw = (nblk + kLeanWorkerWarps - 1u) / kLeanWorkerWarps;   // (the last row of blocks may be partial)
    static_assert((kLeanRing + 2) * kLeanSlotVox * 16 >= 4096 * 4, "set-up scratch: one word per region");
    unsigned* const cursor = BIG ? A.big_cursor : reinterpret_cast<unsigned*>(sm.stage);   // scratch: ring + private stages are idle until the first merge
    for (unsigned s = tid; s < S; s += kFastThreads) {
        const unsigned r0 = A.run_start[s];
        sm.rs[s] = r0; sm.rlen[s] = (unsigned short)(A.run_end[s] - r0); sm.n[s] = R.n[s];
        const int h = R.head[s], t = R.tail[s], nx = R.next_run[s];
        sm.head[s] = (unsigned short)(h < 0 ? kNil16 : (unsigned)h); sm.tail[s] = (unsigned short)(t < 0 ? kNil16 : (unsigned)t);
        sm.next[s] = (unsigned short)(nx < 0 ? kNil16 : (unsigned)nx); sm.mark[s] = (unsigned short)kNil16; sm.adj_start[s] = 0u;
    }
    if (tid < 32) { sm.bdirty[tid] = 1u; sm.wm_key[tid] = kDeadKey64; }      // (lean_head reads 29 partial minima whatever NT is)
    if constexpr (BIG) for (unsigned i = tid; i < (nblk + 31u) / 32u; i += kFastThreads) sm.blkdirty[i] = 0xffffffffu;
    for (int i = tid; i < kLeanMaxTouched; i += kFastThreads) sm.partner[i] = (unsigned short)kNil16;
    for (int i = tid; i < kLeanHash; i += kFastThreads) { sm.hkey[i] = kDeadKey; sm.hcnt[i] = 0u; }
    if constexpr (BIG) {
        const LeanWideScratch ws(reinterpret_cast<char*>(A.big_cursor) + lean_cursor_bytes(A.S_cap));
        for (unsigned i = tid; i < kLeanWideSlots; i += kFastThreads) ws.partner[i] = (unsigned short)kNil16;
        for (unsigned i = tid; i < kLeanWideHash; i += kFastThreads) { ws.hkey[i] = kDeadKey; ws.hcnt[i] = 0u; }
    }
    __syncthreads();
    for (unsigned e = tid; e < A.E_cap; e += kFastThreads) {
        unsigned long long k = kDeadKey64; unsigned ab = kDeadKey;
        if (e < nE && A.E.stamp[e] != kDeadStamp) {
            const float w = A.E.w[e];
            const unsigned hi = isnan(w) ? 0x7f800000u : __float_as_uint(w);
            k = ((unsigned long long)hi << 32) | ((unsigned)(int)A.E.stamp[e] ^ 0x80000000u);
            ab = (A.E.a[e] << 16) | A.E.b[e];
            atomicAdd(&sm.adj_start[ab >> 16], 1u); atomicAdd(&sm.adj_start[ab & 0xffffu], 1u);      // degrees
        }
        sm.key[e] = k; sm.ab[e] = ab;
    }
    if (tid == 0) {
        for (int i = 0; i < 16; ++i) sm.misc[i] = 0;
        sm.misc[FM_EALIVE] = (int)nE; sm.misc[FM_RALIVE] = (int)S; sm.misc[FM_COUNTER] = (int)nE;
        if (A.resume) {
            const MergeCtl* c = A.ctl;
            sm.misc[FM_EALIVE] = (int)c->edges_alive; sm.misc[FM_RALIVE] = (int)c->regions_alive;
            sm.misc[FM_COUNTER] = (int)(c->counter > (long long)nE ? c->counter : (long long)nE);
            sm.misc[FM_NANW] = (int)c->nan_weights; sm.misc[FM_MAXT] = (int)c->max_touched; sm.misc[FM_NMERGES] = (int)c->n_merges;
        }
        for (int i = 0; i < kLeanRing; ++i) { mbar_init(mbar_full + 8u * i, 32u); mbar_init(mbar_empty + 8u * i, 2u); }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    // exclusive scan of the degrees -> list starts (CSR), 1024 regions per round
    for (unsigned base = 0; base < S; base += kFastThreads) {
        const unsigned s = base + tid;
        const unsigned deg = s < S ? sm.adj_start[s] : 0u;
        unsigned incl = deg;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) { const unsigned t = __shfl_up_sync(kFull, incl, off); if (lane >= off) incl += t; }
        if (lane == 31) sm.wm_e[warp] = incl;
        __syncthreads();
        unsigned wpre = 0;
        for (int w = 0; w < warp; ++w) wpre += sm.wm_e[w];
        const unsigned carry = (unsigned)sm.misc[FM_POOL];
        if (s < S) {
            const unsigned st = carry + wpre + incl - deg;
            sm.adj_start[s] = st; cursor[s] = st; sm.adj_len[s] = (unsigned short)deg; sm.adj_cap[s] = (unsigned short)deg;
        }
        __syncthreads();
        if (tid == kFastThreads - 1) sm.misc[FM_POOL] = (int)(carry + wpre + incl);
        __syncthreads();
    }
    if ((unsigned)sm.misc[FM_POOL] > A.pool_cap) { if (tid == 0) sm.misc[FM_ERROR] = (int)kFastErrPool; }
    else
        for (unsigned e = tid; e < A.E_cap; e += kFastThreads) {
            const unsigned ab = sm.ab[e];
            if (ab == kDeadKey) continue;
            adj_pool[atomicAdd(&cursor[ab >> 16], 1u)] = (PoolT)e;
            adj_pool[atomicAdd(&cursor[ab & 0xffffu], 1u)] = (PoolT)e;
        }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // the scratch words become the bulk copies' ring again
    __syncthreads();

    if (warp == 0) {
        // =========== covariance sums + xyz sums: lanes 0..8 each continue one accumulator of region a over b's voxels =====
        const float* stage_f = reinterpret_cast<const float*>(sm.stage);
        const int pi = lane < 3 ? 0 : (lane < 5 ? 1 : (lane == 5 ? 2 : (lane < 9 ? lane - 6 : 0)));
        const int qi = lane < 3 ? lane : (lane < 5 ? lane - 2 : 2);
        const bool prod = lane < 6;
        unsigned chunk = 0;
        LPROF_DECL;
        unsigned nm = 0;                                   // merges so far (trace index)
        while (true) {
            __syncthreads();                                                                   // S1
            const FastHead hd = lean_head(sm, lane);
            LPROF(lane == 0, 3);
            if (sm.misc[FM_ERROR] || hd.hi == kDeadKey || !(__uint_as_float(hd.hi) < A.threshold)) break;
            const unsigned a = hd.ab >> 16, b = hd.ab & 0xffffu;
            if (lean_too_wide<BIG, NT>(sm, a, b)) break;               // more touched edges than worker threads: stop BEFORE this merge (the host continues with the general kernel)
            const int na = sm.n[a], nb = sm.n[b];
            const bool wide = lean_wide(sm, a, b);
            LTRACE(lane == 0, 12, (unsigned)clock()); LTRACE(lane == 0, 21, (unsigned)nb);
            float acc = 0.0f;
            if (lane < 9) {
                const float* src = lane < 4 ? reinterpret_cast<const float*>(R.accu0 + a) + lane
                                 : (lane < 8 ? reinterpret_cast<const float*>(R.accu1 + a) + (lane - 4) : reinterpret_cast<const float*>(R.accu2 + a));
                acc = __ldcg(src);
            }
            const bool direct = nb <= kLeanSlotVox;
            if (direct) lean_fetch_small(sm.head, sm.next, sm.rs, sm.rlen, A.pos_data, b, nb, sm.priv, lane);
            for (int done = 0; done < nb; done += kLeanSlotVox) {
                const int cn = min(nb - done, kLeanSlotVox);
                const unsigned slot = chunk & (kLeanRing - 1);
                if (!direct) mbar_wait(mbar_full + 8u * slot, (chunk / kLeanRing) & 1u);
                LPROF(lane == 0, 0);
                LTRACE(lane == 0 && done == 0, 13, (unsigned)clock());
                const float* sf = direct ? reinterpret_cast<const float*>(sm.priv) : stage_f + slot * (kLeanSlotVox * 4);
                int j = 0;
                for (; j + 8 <= cn; j += 8) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const float p = sf[4 * (j + u) + pi];
                        const float q = prod ? sf[4 * (j + u) + qi] : 1.0f;
                        acc = acc + p * q;
                    }
                }
                for (; j < cn; ++j) {
                    const float p = sf[4 * j + pi];
                    const float q = prod ? sf[4 * j + qi] : 1.0f;
                    acc = acc + p * q;
                }
                if (!direct) {
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(mbar_empty + 8u * slot);
                    ++chunk;
                }
            }
            LPROF(lane == 0, 1);
            LTRACE(lane == 0, 14, (unsigned)clock());
            float cen[3], nv[3], curv;
            plane_from_accu_warp(acc, na + nb, lane, pi, qi, cen, nv, curv);                   // :411-420, spread over the lanes
            const float cx = cen[0], cy = cen[1], cz = cen[2];
            if (lane == 0) {
                sm.newgeo[3] = cx; sm.newgeo[4] = cy; sm.newgeo[5] = cz;
                sm.newgeo[6] = nv[0]; sm.newgeo[7] = nv[1]; sm.newgeo[8] = nv[2];
            }
            __syncwarp();
            LPROF(lane == 0, 2);
            LTRACE(lane == 0, 15, (unsigned)clock());
            if (wide) named_bar(BAR_F, kFastThreads); else named_bar(BAR_FN, 128);              // F: workers read x's old state before this
            if (lane == 0) { R.centroid[a] = make_float4(cx, cy, cz, 0.0f); R.normal[a] = make_float4(nv[0], nv[1], nv[2], curv); }
            if (lane < 9) {                                                                     // every lane stores its own raw sum
                float* dst = lane < 4 ? reinterpret_cast<float*>(R.accu0 + a) + lane
                           : (lane < 8 ? reinterpret_cast<float*>(R.accu1 + a) + (lane - 4) : reinterpret_cast<float*>(R.accu2 + a));
                *dst = acc;
            }
            ++nm;
        }
        LPROF_STORE(lane == 0, 16, 4);
    } else if (warp == 1) {
        // =========== ColorUtilities::mean_color continued: lanes 0..2 carry r, g, b; every lane prepares one reciprocal =====
        const unsigned* stage_u = reinterpret_cast<const unsigned*>(sm.stage);
        const int shift = lane < 3 ? 16 - 8 * lane : 0;
        const EdgeParams ep = A.ep;
        float* const inv_s = sm.inv;
        unsigned chunk = 0;
        unsigned long long fold_steps = A.resume ? A.ctl->fold_steps : 0ull;
        LPROF_DECL;
        unsigned nm = 0;                                   // merges so far (trace index)
        while (true) {
            __syncthreads();                                                                   // S1
            const FastHead hd = lean_head(sm, lane);
            LPROF(lane == 0, 3);
            if (sm.misc[FM_ERROR] || hd.hi == kDeadKey || !(__uint_as_float(hd.hi) < A.threshold)) break;
            const unsigned a = hd.ab >> 16, b = hd.ab & 0xffffu;
            if (lean_too_wide<BIG, NT>(sm, a, b)) break;               // more touched edges than worker threads: stop BEFORE this merge (the host continues with the general kernel)
            const int na = sm.n[a], nb = sm.n[b];
            const bool wide = lean_wide(sm, a, b);
            LTRACE(lane == 0, 16, (unsigned)clock());
            float m = 0.0f, mb_ = 0.0f;
            if (lane < 3) { m = __ldcg(reinterpret_cast<const float*>(R.mean + a) + 1 + lane); mb_ = __ldcg(reinterpret_cast<const float*>(R.mean + b) + 1 + lane); }
            // GUESS of the merged region's colour vector for the workers' speculative colour deltas: the Lab lattice point of the
            // size-weighted mean of the two running means.  It differs from the exact continued running mean by rounding noise
            // only, and OpenCV's LUT quantises its input to 9 bits per channel, so the guess is wrong about once in 10^3 merges
            // (checked against the exact result below; a wrong guess costs a re-evaluation, never a wrong result).
            float guess[3];
            {
                const float gm = (m * (float)na + mb_ * (float)nb) / (float)(na + nb);
                const float gr = __shfl_sync(kFull, gm, 0), gg = __shfl_sync(kFull, gm, 1), gb = __shfl_sync(kFull, gm, 2);
                if (ep.color_mode == 0) rgb2lab_lanes(ep.lab_lut, gr, gg, gb, lane, guess);
                else { guess[0] = gr; guess[1] = gg; guess[2] = gb; }
                if (lane == 0) { sm.newgeo[10] = guess[0]; sm.newgeo[11] = guess[1]; sm.newgeo[12] = guess[2]; }
                __syncwarp();
                if (wide) bar_arrive(BAR_G, 32 + kFastOwners); else bar_arrive(BAR_GN, 64);     // G: guess published
            }
            LPROF(lane == 0, 3);
            LTRACE(lane == 0, 17, (unsigned)clock());
            const float cnt0 = (float)na;
            const bool direct = nb <= kLeanSlotVox;
            if (direct) lean_fetch_small(sm.head, sm.next, sm.rs, sm.rlen, A.pos_data, b, nb, sm.priv + kLeanSlotVox, lane);
            for (int done = 0; done < nb; done += kLeanSlotVox) {
                const int cn = min(nb - done, kLeanSlotVox);
                const unsigned slot = chunk & (kLeanRing - 1);
                float inv_next = 1 / (cnt0 + (float)(done + lane + 1));
                if (!direct) mbar_wait(mbar_full + 8u * slot, (chunk / kLeanRing) & 1u);
                LPROF(lane == 0, 0);
                LTRACE(lane == 0 && done == 0, 18, (unsigned)clock());
                const unsigned* su = direct ? reinterpret_cast<const unsigned*>(sm.priv + kLeanSlotVox) : stage_u + slot * (kLeanSlotVox * 4);
                for (int base = 0, g = 0; base < cn; base += 32, g ^= 1) {
                    inv_s[g * 32 + lane] = inv_next;                       // 1/k of the next 32 voxels, one division per lane
                    inv_next = 1 / (cnt0 + (float)(done + base + 32 + lane + 1));
                    __syncwarp();
                    const int mcount = min(32, cn - base);
                    const float* iv = inv_s + g * 32;
                    const unsigned* sv = su + 4 * base + 3;
#pragma unroll 8
                    for (int j = 0; j < mcount; ++j) {
                        const float x = (float)((sv[4 * j] >> shift) & 255u);
                        m = m + iv[j] * (x - m);
                    }
                }
                if (!direct) {
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(mbar_empty + 8u * slot);
                    ++chunk;
                }
            }
            LPROF(lane == 0, 1);
            LTRACE(lane == 0, 19, (unsigned)clock());
            const float mr = __shfl_sync(kFull, m, 0), mg = __shfl_sync(kFull, m, 1), mb = __shfl_sync(kFull, m, 2);
            float cv[3];
            if (ep.color_mode == 0) rgb2lab_lanes(ep.lab_lut, mr, mg, mb, lane, cv);
            else { cv[0] = mr; cv[1] = mg; cv[2] = mb; }
            if (lane == 0) {
                sm.newgeo[0] = cv[0]; sm.newgeo[1] = cv[1]; sm.newgeo[2] = cv[2];
                newgeo_i[9] = (__float_as_uint(cv[0]) == __float_as_uint(guess[0]) && __float_as_uint(cv[1]) == __float_as_uint(guess[1]) &&
                               __float_as_uint(cv[2]) == __float_as_uint(guess[2])) ? 1 : 0;
            }
            __syncwarp();
            LPROF(lane == 0, 2);
            LTRACE(lane == 0, 20, (unsigned)clock());
            if (wide) named_bar(BAR_F, kFastThreads); else named_bar(BAR_FN, 128);              // F: the workers read the guess before this
            if (lane == 0) {
                R.mean[a] = make_float4((float)(na + nb), mr, mg, mb);
                R.cvec[a] = make_float4(cv[0], cv[1], cv[2], 0.0f);
            }
            fold_steps += (unsigned long long)nb; ++nm;
        }
        if (lane == 0) A.ctl->fold_steps = fold_steps;
        LPROF_STORE(lane == 0, 12, 4);
    } else if (warp == 2) {
        // =========== loader: walk b's rope, copy its runs into the ring (long regions only); splice the ropes =====
        const unsigned stage_addr = smem_addr(sm.stage);
        unsigned chunk = 0;
        while (true) {
            __syncthreads();                                                                   // S1
            const FastHead hd = lean_head(sm, lane);
            if (sm.misc[FM_ERROR] || hd.hi == kDeadKey || !(__uint_as_float(hd.hi) < A.threshold)) break;
            const unsigned a = hd.ab >> 16, b = hd.ab & 0xffffu;
            if (lean_too_wide<BIG, NT>(sm, a, b)) break;               // more touched edges than worker threads: stop BEFORE this merge (the host continues with the general kernel)
            const int na = sm.n[a], nb = sm.n[b];
            const bool wide = lean_wide(sm, a, b);
            if (nb > kLeanSlotVox) {                       // (the fold warps fetch a small region themselves, lean_fetch_small)
                // every lane copies one voxel of the current run per step (16-byte cp.async); a lane's copies of a chunk complete
                // its arrival on the slot's "full" barrier (cp.async.mbarrier.arrive.noinc, 32 arrivals per phase)
                unsigned run = sm.head[b];
                unsigned pos = run != kNil16 ? sm.rs[run] : 0u, end = run != kNil16 ? pos + sm.rlen[run] : 0u;
                for (int done = 0; done < nb; done += kLeanSlotVox, ++chunk) {
                    const int cn = min(nb - done, kLeanSlotVox);
                    const unsigned slot = chunk & (kLeanRing - 1);
                    mbar_wait(mbar_empty + 8u * slot, ((chunk / kLeanRing) & 1u) ^ 1u);           // both fold warps are done with the slot
                    const unsigned dst = stage_addr + slot * (kLeanSlotVox * 16u);
                    int off = 0;
                    while (off < cn && run != kNil16) {
                        const int take = min((int)(end - pos), cn - off);
                        for (int j = lane; j < take; j += 32) cp_async16(dst + (unsigned)(off + j) * 16u, A.pos_data + pos + j);
                        off += take; pos += (unsigned)take;
                        if (pos == end) { run = sm.next[run]; if (run != kNil16) { pos = sm.rs[run]; end = pos + sm.rlen[run]; } }
                    }
                    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(mbar_full + 8u * slot) : "memory");
                }
            }
            if (wide) named_bar(BAR_F, kFastThreads); else named_bar(BAR_FN, 128);              // F
            // rope splice and sizes (voxels_ = a ++ b, :406-409, :426-429) once nobody reads the old ones any more
            if (lane == 0) {
                sm.next[sm.tail[a]] = sm.head[b]; sm.tail[a] = sm.tail[b];
                sm.n[a] = na + nb; sm.n[b] = 0;
            }
        }
    } else {
        // =========== workers: the weight map (cached block minima, adjacency lists) and one touched edge per thread =====
        EdgeParams ep = A.ep;
        if (A.lambda_dev) ep.lambda = *A.lambda_dev;
        const int wtid = tid - 32 * kLeanRoleWarps;                                            // 0..927
        const int ww = warp - kLeanRoleWarps;                                                  // 0..28
        const PoolT* const pool = adj_pool;
        unsigned my_hs = kNil16;                                                               // tie-hash slot to clear after the next S1
        unsigned n_merges = A.resume ? A.ctl->n_merges : 0u;          // (the log continues behind the merges already replayed)
        LPROF_DECL;
        unsigned nm = 0;                                   // merges so far (trace index)
        unsigned long long cls_cyc[4] = {0, 0, 0, 0}; unsigned cls_cnt[4] = {0, 0, 0, 0}; unsigned t_top = 0;   // PROF: merges by touched-edge class
#define WPROF(i) LPROF(wtid == 0, i)
        while (true) {
            if (PROF) t_top = (unsigned)clock();
            LTRACE(wtid == 0, 0, t_top);
            // ---- A: a warp that holds a re-weighted (or removed) edge rescans its blocks (lane l: edge 32 blk + l, the loads
            //         independent) and republishes its minimum ----
            if (sm.bdirty[ww]) {
                __syncwarp();
                if (lane == 0) sm.bdirty[ww] = 0u;
                if constexpr (BIG) {
                    // blocks of this warp whose MINIMUM edge was re-weighted upwards or removed (every other re-weighted edge went into
                    // its block's cached minimum by atomicMin, phase E): the lanes test 32 blocks at a time, the dirty ones are reloaded
                    // (one coalesced 256 + 128-byte load each, eight in flight) and reduced to a new block minimum
                    for (unsigned jb = 0; jb < nbw; jb += 32u) {
                        const unsigned jl = jb + (unsigned)lane, bl = (unsigned)ww + kLeanWorkerWarps * jl;
                        unsigned m = __ballot_sync(kFull, jl < nbw && bl < nblk && ((sm.blkdirty[bl >> 5] >> (bl & 31u)) & 1u));
                        while (m) {
                            unsigned long long k8[8]; unsigned a8[8], b8[8]; bool d8[8];
#pragma unroll
                            for (int u = 0; u < 8; ++u) {
                                d8[u] = m != 0u;
                                const unsigned q = d8[u] ? (unsigned)__ffs(m) - 1u : 0u;
                                m &= m - 1u;
                                b8[u] = (unsigned)ww + kLeanWorkerWarps * (jb + q);
                                k8[u] = d8[u] ? __ldcg(sm.key + b8[u] * 32u + (unsigned)lane) : kDeadKey64;
                                a8[u] = d8[u] ? __ldcg(sm.ab + b8[u] * 32u + (unsigned)lane) : kDeadKey;
                            }
#pragma unroll
                            for (int u = 0; u < 8; ++u) {
                                if (!d8[u]) continue;                                       // (warp-uniform)
                                const unsigned hi = (unsigned)(k8[u] >> 32), lo = (unsigned)k8[u];
                                const unsigned m_hi = __reduce_min_sync(kFull, hi);
                                const unsigned m_lo = __reduce_min_sync(kFull, hi == m_hi ? lo : kDeadKey);
                                if (lane == __ffs(__ballot_sync(kFull, hi == m_hi && lo == m_lo)) - 1) {
                                    sm.bm_key[b8[u]] = k8[u]; sm.bm_e[b8[u]] = b8[u] * 32u + (unsigned)lane; sm.bm_ab[b8[u]] = a8[u];
                                    atomicAnd(&sm.blkdirty[b8[u] >> 5], ~(1u << (b8[u] & 31u)));
                                }
                            }
                        }
                    }
                    __syncwarp();
                    unsigned long long best = kDeadKey64; unsigned bb = 0;
                    for (unsigned j = (unsigned)lane; j < nbw; j += 32u) {
                        const unsigned blk = (unsigned)ww + kLeanWorkerWarps * j;
                        if (blk < nblk) { const unsigned long long k = sm.bm_key[blk]; if (k < best) { best = k; bb = blk; } }
                    }
                    const unsigned hi = (unsigned)(best >> 32), lo = (unsigned)best;
                    const unsigned m_hi = __reduce_min_sync(kFull, hi);
                    const unsigned m_lo = __reduce_min_sync(kFull, hi == m_hi ? lo : kDeadKey);
                    if (lane == __ffs(__ballot_sync(kFull, hi == m_hi && lo == m_lo)) - 1) { sm.wm_key[ww] = best; sm.wm_e[ww] = sm.bm_e[bb]; sm.wm_ab[ww] = sm.bm_ab[bb]; }
                } else {
                unsigned long long best = kDeadKey64; unsigned be = 0;
#pragma unroll 4
                for (unsigned j = 0; j < nbw; ++j) {
                    const unsigned blk = (unsigned)ww + kLeanWorkerWarps * j;
                    const unsigned e = blk * 32u + (unsigned)lane;
                    const unsigned long long k = blk < nblk ? sm.key[e] : kDeadKey64;
                    if (k < best) { best = k; be = e; }
                }
                const unsigned hi = (unsigned)(best >> 32), lo = (unsigned)best;
                const unsigned m_hi = __reduce_min_sync(kFull, hi);
                const unsigned m_lo = __reduce_min_sync(kFull, hi == m_hi ? lo : kDeadKey);
                if (lane == __ffs(__ballot_sync(kFull, hi == m_hi && lo == m_lo)) - 1) { sm.wm_key[ww] = best; sm.wm_e[ww] = be; sm.wm_ab[ww] = sm.ab[be]; }
                }
            }
            WPROF(0);
            LTRACE(wtid == 0, 1, (unsigned)clock());
            __syncthreads();                                                                   // S1
            const FastHead hd = lean_head(sm, lane);
            if (my_hs != kNil16) { sm.hkey[my_hs] = kDeadKey; sm.hcnt[my_hs] = 0u; my_hs = kNil16; }
            if (sm.misc[FM_ERROR] || hd.hi == kDeadKey || !(__uint_as_float(hd.hi) < A.threshold)) break;   // strict <, src/clustering.cpp:388-389
            const unsigned a = hd.ab >> 16, b = hd.ab & 0xffffu;
            if (lean_too_wide<BIG, NT>(sm, a, b)) { if (wtid == 0) sm.misc[FM_ERROR] = (int)kFastErrTouched; break; }   // nothing of this merge has happened yet
            const int counter = sm.misc[FM_COUNTER];
            const unsigned pool_top = (unsigned)sm.misc[FM_POOL];
            WPROF(1);
            LTRACE(wtid == 0, 2, (unsigned)clock());
            // ---- B: the edges incident to a or b come from the two adjacency lists (thread i: entry i) ----
            const unsigned la = sm.adj_len[a], lb = sm.adj_len[b], sa = sm.adj_start[a], sb = sm.adj_start[b];
            const unsigned ca = sm.adj_cap[a], cb = sm.adj_cap[b];
            const int T = (int)(la + lb);
            const bool overflow = T > kLeanMaxTouched;
            const bool wide = T > 32;                                                          // more than one warp of entries
            if (wtid == 0) {
                sm.key[hd.e] = kDeadKey64; sm.ab[hd.e] = kDeadKey;                             // the head edge leaves the map
                const unsigned hb = hd.e >> 5;
                sm.bdirty[hb % kLeanWorkerWarps] = 1u;
                if constexpr (BIG) atomicOr(&sm.blkdirty[hb >> 5], 1u << (hb & 31u));
                if (n_merges < A.log_cap) {                                                    // debug line of :390-392 (ranks; labels at the end)
                    A.mlog.a[n_merges] = a; A.mlog.b[n_merges] = b; A.mlog.w[n_merges] = __uint_as_float(hd.hi);
                    A.mlog.edges_left[n_merges] = (unsigned)sm.misc[FM_EALIVE]; A.mlog.regions_left[n_merges] = (unsigned)sm.misc[FM_RALIVE];
                }
            }
            if constexpr (BIG) {
                if (T > kLeanMaxTouched) {                 // more adjacency entries than worker threads (CTA-uniform): every thread loops
                    lean_wide_merge<PROF>(A, ep.lambda, hd.e, a, b, counter, pool_top, wtid);
                    named_bar(BAR_W4, kFastOwners);                                            // W4
                    WPROF(7);
                    if (PROF && wtid == 0) { cls_cyc[3] += (unsigned)clock() - t_top; cls_cnt[3]++; }
                    ++n_merges; ++nm;
                    continue;
                }
            }
            // ---- C: duplicates (a,x)/(b,x) through a per-region mark; x's geometry; speculative colour deltas ----
            // Colour deltas are memoised per edge and speculated: while the fold runs, the edges whose stored delta does not
            // fit the GUESS of the merged region's colour vector (warp 1: Lab lattice point of the size-weighted mean) get
            // CIEDE2000 against the guess.  A wrong guess (about 1 merge in 10^3) re-evaluates after the fold.
            unsigned e = 0, x = 0; bool side_a = false, mine = false; unsigned long long okey = kDeadKey64, nkey = kDeadKey64;
            bool live = false, need = false;
            float dc = 0.0f; float4 xcv, c4, n4, ocv;
            const bool active = ww == 0 || wide;
            if (active) {
                if (!overflow && wtid < T) {
                    e = __ldcg(pool + ((unsigned)wtid < la ? sa + (unsigned)wtid : sb + ((unsigned)wtid - la)));
                    const unsigned eab = sm.ab[e];
                    mine = e != hd.e && eab != kDeadKey;                                       // lists keep removed edges until they are rewritten
                    if (mine) {
                        okey = sm.key[e]; sm.te_key[wtid] = okey;
                        const unsigned ea = eab >> 16, eb = eab & 0xffffu;
                        side_a = ea == a || eb == a;
                        x = (ea == a || ea == b) ? eb : ea;
                        const unsigned short old = atomicCAS(&sm.mark[x], (unsigned short)kNil16, (unsigned short)wtid);
                        if (old != (unsigned short)kNil16) { sm.partner[wtid] = old; sm.partner[old] = (unsigned short)wtid; }
                        xcv = __ldcg(R.cvec + x); c4 = __ldcg(R.centroid + x); n4 = __ldcg(R.normal + x); dc = __ldcg(A.E.dc + e);
                        ocv = __ldcg(R.cvec + (side_a ? a : b));                               // the colour vector the stored delta was computed with
                    }
                }
                if (wide) named_bar(BAR_WB, kFastOwners); else __syncwarp();                   // WB1
            }
            WPROF(2);
            LTRACE(wtid == 0, 3, (unsigned)clock()); LTRACE(wtid == 0, 8, (unsigned)T);
            if (wide) named_bar(BAR_G, 32 + kFastOwners); else if (active) named_bar(BAR_GN, 64);   // G: the guess of a's new colour vector
            const float4 guess = make_float4(sm.newgeo[10], sm.newgeo[11], sm.newgeo[12], 0.0f);
            if (mine) {
                const unsigned q = sm.partner[wtid];
                const bool dup = q != kNil16 && sm.te_key[q] < okey;                           // the earlier of (a,x), (b,x) survives
                sm.mark[x] = (unsigned short)kNil16; sm.partner[wtid] = (unsigned short)kNil16;
                live = !dup;
                // the stored delta stays valid when the end that changes keeps its colour vector and the argument order
                const bool same_cv = __float_as_uint(ocv.x) == __float_as_uint(guess.x) && __float_as_uint(ocv.y) == __float_as_uint(guess.y) &&
                                     __float_as_uint(ocv.z) == __float_as_uint(guess.z);
                const bool reuse = same_cv && (side_a || ((b < x) == (a < x)));
                need = live && !reuse;
                if (need) { const bool af = a < x; dc = colour_delta(ep.color_mode, af ? guess : xcv, af ? xcv : guess); }   // ONE call site: lanes must not diverge around 800 instructions
            }
            WPROF(3);
            LTRACE(wtid == 0, 4, (unsigned)clock());
            if (wide) named_bar(BAR_F, kFastThreads); else if (active) named_bar(BAR_FN, 128);  // F: region a's new colour vector / centroid / normal
            WPROF(4);
            LTRACE(wtid == 0, 5, (unsigned)clock());
            // ---- D: colour delta after a wrong guess, geometry delta, weight, classification, tie stamps, a's new list ----
            // a's new adjacency list goes into a's block, else into b's, else into a fresh one twice the size (T bounds the survivors)
            const bool fresh = ca < (unsigned)T && cb < (unsigned)T;
            const unsigned ncap = fresh ? min(2u * (unsigned)T, 65535u) : (ca >= (unsigned)T ? ca : cb);
            const unsigned dst = ca >= (unsigned)T ? sa : (cb >= (unsigned)T ? sb : pool_top);
            const bool pool_ok = !fresh || pool_top + ncap <= A.pool_cap;
            if (active) {
                unsigned wbits = kDeadKey, nab = kDeadKey; int cls = FC_DUP; unsigned hs = kNil16;
                const bool hit = newgeo_i[9] != 0;
                // a's new adjacency list: in a's block, else in b's, else a fresh one twice the size (T bounds the survivors)
                if (mine) {
                    const bool redo = !hit && live;                                            // wrong guess (rare): every survivor re-evaluates
                    if (redo) {
                        const float4 acv = make_float4(sm.newgeo[0], sm.newgeo[1], sm.newgeo[2], 0.0f);
                        const bool af = a < x;
                        dc = colour_delta(ep.color_mode, af ? acv : xcv, af ? xcv : acv);
                    }
                    if (PROF && (redo || need)) atomicAdd(&sm.misc[FM_EVALS], (redo ? 1 : 0) + (need ? 1 : 0));
                    if (live) {
                        const float4 ace = make_float4(sm.newgeo[3], sm.newgeo[4], sm.newgeo[5], 0.0f), anr = make_float4(sm.newgeo[6], sm.newgeo[7], sm.newgeo[8], 0.0f);
                        const bool a_first = a < x;
                        const float dg = geom_delta(ep.geom_mode, a_first ? anr : n4, a_first ? ace : c4, a_first ? n4 : anr, a_first ? c4 : ace);
                        nab = a_first ? (a << 16) | x : (x << 16) | a;
                        float w_new = unify(ep, dc, dg);
                        if (isnan(w_new)) { atomicAdd(&sm.misc[FM_NANW], 1); w_new = __int_as_float(0x7f800000); }
                        wbits = __float_as_uint(w_new);
                        const unsigned old_hi = (unsigned)(okey >> 32);
                        cls = wbits == old_hi ? FC_KEEP : (wbits > old_hi ? FC_FRONT : FC_BACK);
                        if (cls != FC_KEEP && wide) {                                          // tie groups: same new weight, same side
                            const unsigned hk = wbits | (cls == FC_FRONT ? 0x80000000u : 0u);
                            unsigned h = (hk * 2654435761u) >> kLeanHashShift;
                            while (true) {
                                const unsigned prev = atomicCAS(&sm.hkey[h], kDeadKey, hk);
                                if (prev == kDeadKey || prev == hk) break;
                                h = (h + 1) & (kLeanHash - 1);
                            }
                            atomicAdd(&sm.hcnt[h], 1u);
                            hs = h;
                        }
                        A.E.dc[e] = dc;
                    } else if (wide) atomicAdd(&sm.misc[FM_ND], 1);
                    sm.res_w[wtid] = wbits; sm.cls[wtid] = (unsigned char)cls;
                } else if (!overflow && wtid < T) { sm.res_w[wtid] = kDeadKey; sm.cls[wtid] = (unsigned char)FC_DUP; }   // a removed edge's entry
                unsigned narrow_rank = 0, narrow_gsz = 1;
                {   // survivors take consecutive places in a's new list
                    const unsigned lm = __ballot_sync(kFull, live), mm = __ballot_sync(kFull, mine);
                    int base = 0;
                    if (wide) {
                        const int leader = __ffs(lm) - 1;
                        if (lm && lane == leader) base = atomicAdd(&sm.misc[FM_NLIVE], __popc(lm));
                        base = __shfl_sync(kFull, base, leader < 0 ? 0 : leader);
                    } else {
                        if (lane == 0) { sm.misc[FM_NLIVE] = __popc(lm); sm.misc[FM_ND] = __popc(mm & ~lm); }
                        // one warp holds every touched edge: tie groups by match, ranks by the old keys of the group's lanes
                        const unsigned hk = (live && cls != FC_KEEP) ? (wbits | (cls == FC_FRONT ? 0x80000000u : 0u)) : (0xffffff00u | (unsigned)lane);
                        unsigned grp = __match_any_sync(kFull, hk);
                        narrow_gsz = (unsigned)__popc(grp);
                        if (narrow_gsz > 1) {                                                  // (whole groups take this branch together)
                            grp &= ~(1u << lane);
                            while (grp) { const int q = __ffs(grp) - 1; grp &= grp - 1u; if (sm.te_key[(wtid & ~31) + q] < okey) ++narrow_rank; }
                        }
                    }
                    if (live && pool_ok) adj_pool[dst + (unsigned)base + (unsigned)__popc(lm & ((1u << lane) - 1u))] = (PoolT)e;
                }
                if (wide) named_bar(BAR_WB, kFastOwners); else __syncwarp();                   // WB2
                if (mine) {
                    unsigned lo = (unsigned)okey;
                    if (!wide) {
                        if (live && cls != FC_KEEP) {
                            const int st = cls == FC_BACK ? counter + (int)narrow_rank : -(counter + (int)(narrow_gsz - 1 - narrow_rank));
                            lo = (unsigned)st ^ 0x80000000u;
                        }
                    } else if (hs != kNil16) {
                        const unsigned gsz = sm.hcnt[hs];
                        unsigned rank = 0;
                        if (gsz > 1)                                                           // new arrivals keep their old relative order inside a tie group
#pragma unroll 1
                            for (int q = 0; q < T; ++q)
                                if (sm.cls[q] == cls && sm.res_w[q] == wbits && sm.te_key[q] < okey) ++rank;
                        const int st = cls == FC_BACK ? counter + (int)rank : -(counter + (int)(gsz - 1 - rank));
                        lo = (unsigned)st ^ 0x80000000u;
                        my_hs = hs;
                    }
                    nkey = live ? ((unsigned long long)wbits << 32) | lo : kDeadKey64;
                    sm.key[e] = nkey;
                    sm.ab[e] = nab;
                    sm.bdirty[(e >> 5) % kLeanWorkerWarps] = 1u;
                    if constexpr (BIG) lean_block_min_update(sm, e, okey, nkey);
                }
                if constexpr (BIG) {                                                           // the new block minima's edge / end points
                    if (wide) named_bar(BAR_WB, kFastOwners); else __syncwarp();
                    if (mine && live && sm.bm_key[e >> 5] == nkey) { sm.bm_e[e >> 5] = e; sm.bm_ab[e >> 5] = nab; }
                }
            }
            if (wtid == 0) {
                if (overflow) sm.misc[FM_ERROR] = (int)kFastErrTouched;                        // the host falls back to merge_kernel
                else {
                    if (counter > 0x7f000000 - T) sm.misc[FM_ERROR] = (int)kFastErrStamp;
                    if (!pool_ok) sm.misc[FM_ERROR] = (int)kFastErrPool;
                    else if (fresh) sm.misc[FM_POOL] = (int)(pool_top + ncap);
                    sm.adj_start[a] = dst;
                    sm.adj_len[a] = (unsigned short)sm.misc[FM_NLIVE]; sm.adj_cap[a] = (unsigned short)ncap; sm.adj_len[b] = 0; sm.adj_cap[b] = 0;
                    sm.misc[FM_NLIVE] = 0;
                    sm.misc[FM_COUNTER] = counter + T;
                    sm.misc[FM_EALIVE] -= 1 + sm.misc[FM_ND]; sm.misc[FM_ND] = 0; sm.misc[FM_RALIVE] -= 1;
                    if (T > sm.misc[FM_MAXT]) sm.misc[FM_MAXT] = T;
                    sm.misc[FM_SUMT] += T; sm.misc[FM_MISS] += newgeo_i[9] ? 0 : 1;
                }
            }
            WPROF(5);
            LTRACE(wtid == 0, 6, (unsigned)clock());
            named_bar(BAR_W4, kFastOwners);                                                    // W4: new keys and a's list written
            WPROF(6);
            LTRACE(wtid == 0, 7, (unsigned)clock());
            if (PROF && wtid == 0) { const int c_ = T <= 32 ? 0 : (T <= 128 ? 1 : 2); cls_cyc[c_] += (unsigned)clock() - t_top; cls_cnt[c_]++; }
            ++n_merges; ++nm;
        }
#undef WPROF
        LPROF_STORE(wtid == 0, 0, 8);
        if (PROF && wtid == 0) for (int i = 0; i < 4; ++i) { A.ctl->phase_cycles[8 + i] = cls_cyc[i]; A.ctl->phase_cycles[i < 3 ? 28 + i : 31] = cls_cnt[i]; }
        if (wtid == 0) sm.misc[FM_NMERGES] = (int)n_merges;
    }

    // ---- write back: weight map, ropes, log labels, counters ---------------------------------------------------------
    __syncthreads();
    const unsigned n_merges = (unsigned)sm.misc[FM_NMERGES];
    for (unsigned e = tid; e < nE; e += kFastThreads) {
        const unsigned long long k = sm.key[e];
        if (k == kDeadKey64) A.E.stamp[e] = kDeadStamp;
        else {
            const unsigned ab = sm.ab[e];
            A.E.a[e] = ab >> 16; A.E.b[e] = ab & 0xffffu; A.E.w[e] = __uint_as_float((unsigned)(k >> 32));
            A.E.stamp[e] = (long long)(int)((unsigned)k ^ 0x80000000u);
        }
    }
    for (unsigned s = tid; s < S; s += kFastThreads) {
        R.n[s] = sm.n[s];
        R.head[s] = sm.head[s] == kNil16 ? -1 : (int)sm.head[s]; R.tail[s] = sm.tail[s] == kNil16 ? -1 : (int)sm.tail[s];
        R.next_run[s] = sm.next[s] == kNil16 ? -1 : (int)sm.next[s];
    }
    for (unsigned m = nm_first + tid; m < n_merges && m < A.log_cap; m += kFastThreads) { A.mlog.a[m] = A.sv_label[A.mlog.a[m]]; A.mlog.b[m] = A.sv_label[A.mlog.b[m]]; }   // ranks -> labels, this launch's entries
    if (tid == 0) {
        MergeCtl* ctl = A.ctl;
        ctl->phase_cycles[24] = (unsigned long long)sm.misc[FM_MISS]; ctl->phase_cycles[25] = (unsigned long long)sm.misc[FM_EVALS];
        ctl->phase_cycles[27] = (unsigned long long)sm.misc[FM_SUMT];
        ctl->n_merges = n_merges; ctl->edges_alive = (unsigned)sm.misc[FM_EALIVE]; ctl->regions_alive = (unsigned)sm.misc[FM_RALIVE];
        ctl->counter = (long long)sm.misc[FM_COUNTER];
        ctl->max_touched = (unsigned)sm.misc[FM_MAXT]; ctl->nan_weights = (unsigned)sm.misc[FM_NANW]; ctl->error = (unsigned)sm.misc[FM_ERROR];
    }
}

// one frame: one CTA
template <bool PROF, int NT>
__global__ void __launch_bounds__(NT, 1) merge_fast_kernel(const __grid_constant__ FastArgs A) { merge_lean_body<PROF, false, NT>(A); }
constexpr int kFastThreadsSolo = 768;                // one frame alone (f3ps_merge); grids of frames keep 1024

// graphs too large for an SM's shared memory (C5-size scenes): the same loop with the big tables in global memory
template <bool PROF>
__global__ void __launch_bounds__(kFastThreads, 1) merge_fast_big_kernel(const __grid_constant__ FastArgs A) { merge_lean_body<PROF, true>(A); }

// A batch of frames in ONE launch, CTA i replays frame i (f3ps.cu: merge_frames).  Independent streams share at most 32 hardware
// queues (CUDA_DEVICE_MAX_CONNECTIONS), so at most 32 single-CTA merge kernels ever overlap; one grid has no such limit.
// The per-frame arguments travel in the kernel parameter space (<= 32,764 bytes on sm_70+ with CUDA >= 12.1).
constexpr int kFastBatchMax = 32764 / (int)sizeof(FastArgs) < 96 ? 32764 / (int)sizeof(FastArgs) : 96;
struct FastBatch { FastArgs a[kFastBatchMax]; };
static_assert(sizeof(FastBatch) <= 32764, "kernel parameter space");
__global__ void __launch_bounds__(kFastThreads, 1) merge_fast_batch_kernel(const __grid_constant__ FastBatch B) { merge_lean_body<false>(B.a[blockIdx.x]); }

// What follows a merge kernel, for every frame of its chunk in launches on the chunk's stream (f3ps.cu: launch_chunk):
// Clustering::get_labeled_cloud (:640-663) of every frame (CTA i / grid row i = frame i), then, for a chunk of several frames,
// their device scalars gathered into one array for a single copy to the host.  The kernels read the arrays through __restrict__
// locals: that lets the compiler load them, owner[] among them, through the non-coherent path.
struct LabelArgs {
    RegionArrays R; const unsigned* n_sv_ptr; const unsigned* run_start; const unsigned* run_end;
    unsigned* run_out_off; unsigned* run_dense; unsigned* region_dense; unsigned* n_out;
    const unsigned* pos_run; unsigned n_pos; const unsigned* order; const float4* vox_xyz;
    float* out_xyz; unsigned* out_label; unsigned* out_voxel; unsigned* vox_segment; const unsigned* pos_label; const unsigned* owner;
    const unsigned* scalars;         // the frame's DevScalars, as words
};
struct LabelBatch { LabelArgs a[kFastBatchMax]; };
static_assert(sizeof(LabelBatch) <= 32764, "kernel parameter space");
// dense labels 0..K-1 in ascending region label order; output offset of every run of every rope.  One block per frame: two
// exclusive scans over the regions (alive flag -> dense label, voxel count -> output offset), then one thread per surviving
// region walks its rope.
__global__ void __launch_bounds__(1024) dense_label_batch_kernel(const __grid_constant__ LabelBatch B) {
    const LabelArgs& A = B.a[blockIdx.x];
    const RegionArrays R = A.R;
    const unsigned* __restrict__ n_sv_ptr = A.n_sv_ptr; const unsigned* __restrict__ run_start = A.run_start;
    const unsigned* __restrict__ run_end = A.run_end; unsigned* __restrict__ run_out_off = A.run_out_off;
    unsigned* __restrict__ run_dense = A.run_dense; unsigned* __restrict__ region_dense = A.region_dense; unsigned* __restrict__ n_out = A.n_out;
    __shared__ unsigned s_wa[32], s_wn[32];
    __shared__ unsigned s_ca, s_cn;
    const unsigned S = *n_sv_ptr;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) { s_ca = 0; s_cn = 0; }
    __syncthreads();
    for (unsigned base = 0; base < S; base += blockDim.x) {
        const unsigned s = base + threadIdx.x;
        const int nv = s < S ? R.n[s] : 0;
        const unsigned alive = nv > 0 ? 1u : 0u, cnt = nv > 0 ? (unsigned)nv : 0u;
        unsigned ia = alive, in = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned ta = __shfl_up_sync(kFull, ia, o), tn = __shfl_up_sync(kFull, in, o);
            if (lane >= o) { ia += ta; in += tn; }
        }
        if (lane == 31) { s_wa[warp] = ia; s_wn[warp] = in; }
        __syncthreads();
        unsigned wa = 0, wn = 0;
        for (int w = 0; w < warp; ++w) { wa += s_wa[w]; wn += s_wn[w]; }
        const unsigned ca = s_ca, cn = s_cn;
        if (s < S) {
            if (!alive) region_dense[s] = 0xffffffffu;
            else {
                const unsigned dense = ca + wa + ia - 1u;
                unsigned off = cn + wn + in - cnt;
                region_dense[s] = dense;
                for (int run = R.head[s]; run >= 0; run = R.next_run[run]) {
                    run_out_off[run] = off; run_dense[run] = dense;
                    off += run_end[run] - run_start[run];
                }
            }
        }
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) { s_ca = ca + wa + ia; s_cn = cn + wn + in; }
        __syncthreads();
    }
    if (threadIdx.x == 0) *n_out = s_cn;
}
__global__ void __launch_bounds__(256) labeled_cloud_batch_kernel(const __grid_constant__ LabelBatch B) {
    const LabelArgs& A = B.a[blockIdx.y];
    const unsigned* __restrict__ pos_run = A.pos_run; const unsigned n_pos = A.n_pos; const unsigned* __restrict__ order = A.order;
    const unsigned* __restrict__ run_start = A.run_start; const unsigned* __restrict__ run_out_off = A.run_out_off;
    const unsigned* __restrict__ run_dense = A.run_dense; const float4* __restrict__ vox_xyz = A.vox_xyz;
    float* __restrict__ out_xyz = A.out_xyz; unsigned* __restrict__ out_label = A.out_label; unsigned* __restrict__ out_voxel = A.out_voxel;
    unsigned* __restrict__ vox_segment = A.vox_segment; const unsigned* __restrict__ pos_label = A.pos_label; const unsigned* __restrict__ owner = A.owner;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pos; i += gridDim.x * blockDim.x) {
        const unsigned run = pos_run[i];
        if (run == 0xffffffffu) continue;                 // unowned voxel: absent from every region
        const unsigned o = run_out_off[run] + (i - run_start[run]);
        const unsigned v = order[i];
        const float4 p = vox_xyz[v];
        out_xyz[3 * (size_t)o] = p.x; out_xyz[3 * (size_t)o + 1] = p.y; out_xyz[3 * (size_t)o + 2] = p.z;
        out_label[o] = run_dense[run]; out_voxel[o] = v;
        if (!owner || owner[v] == pos_label[i]) vox_segment[v] = run_dense[run];   // a phantom leaf does not relabel its voxel
    }
}
__global__ void scalars_gather_kernel(const __grid_constant__ LabelBatch B, unsigned words, unsigned* __restrict__ out) {
    const unsigned* __restrict__ src = B.a[blockIdx.x].scalars;
    for (unsigned w = threadIdx.x; w < words; w += blockDim.x) out[(size_t)blockIdx.x * words + w] = src[w];
}

} // namespace f3ps
