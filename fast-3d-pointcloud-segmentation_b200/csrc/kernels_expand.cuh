// kernels_expand.cuh -- K5: pcl::SupervoxelClustering::createSupervoxelHelpers + expandSupervoxels +
// makeSupervoxels' per-helper voxel lists (SURVEY.md A.5/A.6; call site
// /root/reference/src/supervoxel_clustering.cpp:357) as ONE persistent cooperative kernel.
//
// All expansion rounds run inside a single launch; the CTAs meet at a grid barrier between phases:
//   per round:  sweeps until the steal table is a fixed point   (1 barrier each, ~3 per round)
//               count  -> scan -> fill -> ordered centroid fold (4 barriers)
// The sweep is the exact data-parallel restatement of PCL's sequential helper loop (oracle:
// Oracle::expand_fixed_point): voxel n folds, in ascending label order, every helper that holds a leaf
// adjacent to n at its turn.  "Phantom" leaves (two seed cells elected the same voxel; the earlier helper
// keeps the leaf in its set without owning it) are modelled exactly for up to four seed cells on one voxel
// (three holders + the owner); more are reported as F3PS_ERR_CAPACITY.
//
// Cross-CTA mutable state (owner / dist / steal table / centroids / lists) is read with ld.global.cg
// (L2 is the coherence point) and published with a fence before every barrier arrival.
#pragma once
#include "kernels_vccs.cuh"

namespace f3ps {

constexpr int kPhSlots = 3;                     // helpers that can hold one voxel as a phantom leaf (four seed cells electing one voxel)
constexpr unsigned kOwnMask = 0x0fffffffu;      // label bits of an owner word
constexpr unsigned kOwnPhantom = 0x80000000u;   // voxel is held as a phantom leaf by the helpers phantom[kPhSlots * v + s]
constexpr unsigned kOwnWon = 0x70000000u;       // bit 28 + s: the holder in slot s stole it in the round being evaluated
__device__ __forceinline__ unsigned own_won_bit(int s) { return 0x10000000u << s; }
constexpr int kExpandThreads = 512;
#ifndef F3PS_EXPAND_MIN_BLOCKS
#define F3PS_EXPAND_MIN_BLOCKS 2          // 64 registers per thread: two CTAs per SM hide the latency of the neighbour probes
#endif
constexpr int kExpandMaxSweeps = 32;
constexpr int kMaxCand = 32;

enum { EXPAND_ERR_TRIPLE = 1u, EXPAND_ERR_CAND = 2u, EXPAND_ERR_SWEEPS = 4u };

struct ExpandCtl {
    unsigned bar_count, cursor;       // grid barrier arrivals (monotone); bump cursor of the per-helper leaf lists
    unsigned error;                   // EXPAND_ERR_*
    unsigned sweeps_total;
    unsigned n_sv, n_pos;             // surviving helpers; positions of the helper-ordered voxel list (V + surviving phantoms)
    unsigned pad[2];
    unsigned long long t_phase[8];    // ns per phase (CTA 0's view): init, sweeps, (count), alloc, fill, fold, tail
    unsigned changed[64];             // ring indexed by the running sweep number; entry k+2 is cleared during sweep k
};

struct ExpandArgs {
    // immutable inputs
    const int* nbr_col; const int* nbr_row; unsigned V_cap;
    const float4* vox_xyz; const float4* vox_rgb; const float4* vox_nrm;
    const int* seeds;
    unsigned V, S0; int rounds;
    int keep_centroids;               // refineSupervoxels: the helpers keep their centroids, seeds[i] < 0 = helper i + 1 was erased
    VccsParams P;
    // mutable state
    unsigned* owner[2]; float* dist[2]; unsigned* st[2];
    unsigned char* chg[2];            // per voxel: did its steal-table entry move in the sweep that wrote it (active-set sweeps)
    unsigned* phantom; int* phantom_leaf;
    Centroids cen;
    unsigned* count[2]; unsigned* fill; unsigned* off;         // per label [S0 + 2]
    unsigned* list_raw; unsigned* list_sorted; unsigned* pos_label;   // [V + S0]
    // outputs
    unsigned* labels_out; float* dist_out;
    unsigned* seg_end; unsigned* sv_label; unsigned* rank_of_label;
    ExpandCtl* ctl;
};

__device__ __forceinline__ unsigned ldcg_u(const unsigned* p) { return __ldcg(p); }
__device__ __forceinline__ float ldcg_f(const float* p) { return __ldcg(p); }
__device__ __forceinline__ float4 ldcg_f4(const float4* p) { return __ldcg(p); }

// Grid barrier for a cooperatively launched grid: arrivals only ever count up, so phase k is complete
// when the counter reaches k * nblocks (no reset, no generation word).
__device__ __forceinline__ void grid_barrier(ExpandCtl* ctl, unsigned nblocks, unsigned& phase) {
    ++phase;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(&ctl->bar_count, 1u);
        const unsigned target = phase * nblocks;
        volatile unsigned* c = &ctl->bar_count;
        while (*c < target) { }
        __threadfence();
    }
    __syncthreads();
}

// The same meeting point for a grid that is ONE thread-block cluster (expand_cluster_kernel): the hardware cluster barrier,
// release / acquire at cluster scope (global writes made before the arrival are visible to every CTA of the cluster after
// the wait).  ~0.2 us against ~2.5 us for the L2 counter above.
__device__ __forceinline__ void cluster_barrier() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
template <bool CLUSTER>
__device__ __forceinline__ void expand_barrier(ExpandCtl* ctl, unsigned nblocks, unsigned& phase) {
    if constexpr (CLUSTER) cluster_barrier(); else grid_barrier(ctl, nblocks, phase);
}

__device__ __forceinline__ unsigned long long globaltimer_ns() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define XPHASE(i) do { if (tid == 0) { const unsigned long long t_now = globaltimer_ns(); ctl->t_phase[i] += t_now - t_prev; t_prev = t_now; } } while (0)

// One voxel of one sweep: fold, in ascending label order, every helper that holds a leaf adjacent to n at its turn
// (SupervoxelHelper::expand restated per voxel, SURVEY.md A.5).  Reads the round-start owners / distances and the previous
// sweep's steal table, writes this voxel's entries of the next ones.
//
// Active set: the result for n is a pure function of the round-start state and of the steal-table entries of its
// NEIGHBOURS; when none of them moved in the previous sweep (chg_in), this sweep reproduces the previous one, whose owner /
// distance are still in own1 / dst1 (same buffers for every sweep of a round) -- only the entry is carried over and the
// helper sizes are tallied.  chg_in == nullptr (first sweep of a round): everything is evaluated.
__device__ __forceinline__ void expand_sweep_voxel(const ExpandArgs& A, const unsigned n, const unsigned* own0, const float* dst0,
        unsigned* own1, float* dst1, const unsigned* st_in, unsigned* st_out, unsigned* cnt, unsigned& any_change,
        const unsigned char* chg_in, unsigned char* chg_out) {
    const unsigned w0 = own0[n];
    float D = dst0[n];
    const unsigned st_n = st_in[n];
    const int cnt_n = A.nbr_row[(size_t)n * kNbrStride + 27];
    unsigned cur_l = w0 & kOwnMask;
    unsigned idx[27], hu[27];
    unsigned any_ph = w0 & kOwnPhantom;
#pragma unroll
    for (int r = 0; r < 27; ++r) idx[r] = r < cnt_n ? (unsigned)A.nbr_col[(size_t)r * A.V_cap + n] : n;
    if (chg_in) {
        unsigned moved = 0;
#pragma unroll
        for (int r = 0; r < 27; ++r) moved |= idx[r] != n ? (unsigned)chg_in[idx[r]] : 0u;
        if (!moved) {
            const unsigned w1 = own1[n];                       // what the previous sweep decided
            st_out[n] = st_n;
            chg_out[n] = 0;
            const unsigned l1 = w1 & kOwnMask;
            if (l1) atomicAdd(&cnt[l1], 1u);
            if (w0 & kOwnPhantom)
                for (int s = 0; s < kPhSlots; ++s) { const unsigned h = A.phantom[(size_t)kPhSlots * n + s]; if (h && !(w1 & own_won_bit(s))) atomicAdd(&cnt[h], 1u); }
            return;
        }
    }
#pragma unroll
    for (int r = 0; r < 27; ++r) hu[r] = idx[r] != n ? own0[idx[r]] : 0u;
#pragma unroll
    for (int r = 0; r < 27; ++r) {
        any_ph |= hu[r] & kOwnPhantom;
        const unsigned h = hu[r] & kOwnMask;
        const unsigned stv = h != 0u ? st_in[idx[r]] : 0u;
        hu[r] = stv > h ? h : 0u;                 // still h's leaf at h's turn
    }
    unsigned first = kNoSteal, won = 0u, ph_n[kPhSlots] = {0u, 0u, 0u};
    const float4 vx = A.vox_xyz[n], vc = A.vox_rgb[n], vn = A.vox_nrm[n];
    if (!any_ph) {
        unsigned last = 0u;
        while (true) {                            // distinct candidate labels in ascending order
            unsigned m = 0xffffffffu;
#pragma unroll
            for (int r = 0; r < 27; ++r) { const unsigned h = hu[r]; if (h > last && h < m) m = h; }
            if (m == 0xffffffffu) break;
            last = m;
            if (m == cur_l) continue;
            const float d = voxel_data_distance(A.cen.xyz[m], A.cen.rgb[m], A.cen.nrm[m], vx, vc, vn, A.P);
            if (d < D) { if (first == kNoSteal) first = m; D = d; cur_l = m; }
        }
    } else {
        // a phantom leaf somewhere in the neighbourhood: it supports all its neighbours, itself included
        if (w0 & kOwnPhantom) for (int s = 0; s < kPhSlots; ++s) ph_n[s] = A.phantom[(size_t)kPhSlots * n + s];
        unsigned cand[kMaxCand]; int nc = 0; bool overflow = false;
        auto insert = [&](unsigned h) {           // sorted, distinct
            int p = nc;
            while (p > 0 && cand[p - 1] >= h) { if (cand[p - 1] == h) return; --p; }
            if (nc == kMaxCand) { overflow = true; return; }
            for (int q = nc; q > p; --q) cand[q] = cand[q - 1];
            cand[p] = h; ++nc;
        };
        for (int r = 0; r < cnt_n; ++r) {
            const unsigned u = (unsigned)A.nbr_col[(size_t)r * A.V_cap + n];
            const unsigned wu = (u == n) ? w0 : own0[u];
            if (u != n) {
                const unsigned h = wu & kOwnMask;
                if (h != 0u && st_in[u] > h) insert(h);
            }
            if (wu & kOwnPhantom) for (int s = 0; s < kPhSlots; ++s) { const unsigned h = A.phantom[(size_t)kPhSlots * u + s]; if (h) insert(h); }
        }
        if (overflow) atomicOr(&A.ctl->error, (unsigned)EXPAND_ERR_CAND);
        for (int q = 0; q < nc; ++q) {
            const unsigned h = cand[q];
            if (h == cur_l) continue;
            const float d = voxel_data_distance(A.cen.xyz[h], A.cen.rgb[h], A.cen.nrm[h], vx, vc, vn, A.P);
            if (d < D) {
                if (first == kNoSteal) first = h;
                D = d; cur_l = h;
                for (int s = 0; s < kPhSlots; ++s) if (h == ph_n[s]) won |= own_won_bit(s);
            }
        }
    }
    own1[n] = cur_l | (w0 & kOwnPhantom) | won; dst1[n] = D; st_out[n] = first;
    if (chg_out) chg_out[n] = first != st_n ? 1 : 0;
    if (first != st_n) any_change = 1;
    if (cur_l) atomicAdd(&cnt[cur_l], 1u);
    for (int s = 0; s < kPhSlots; ++s) if (ph_n[s] && !(won & own_won_bit(s))) atomicAdd(&cnt[ph_n[s]], 1u);   // a holder that did not steal it still lists its phantom leaf
}

// one contiguous leaf list per helper: 32 helpers per warp, warp-aggregated bump allocation (helper order is irrelevant)
__device__ __forceinline__ void expand_alloc_warp(const ExpandArgs& A, const unsigned* cnt_final, const unsigned base, const int lane) {
    const unsigned l = base + lane + 1u;
    const unsigned c = l <= A.S0 ? cnt_final[l] : 0u;
    unsigned incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { unsigned t = __shfl_up_sync(kFull, incl, o); if (lane >= o) incl += t; }
    unsigned start = 0u;
    if (lane == 31 && incl) start = atomicAdd(&A.ctl->cursor, incl);
    start = __shfl_sync(kFull, start, 31);
    if (l <= A.S0) { A.off[l] = start + incl - c; A.fill[l] = 0u; }
}

// commit the round for voxel n (a phantom leaf its holder stole becomes a regular leaf) and append it to its helpers' lists
__device__ __forceinline__ void expand_fill_voxel(const ExpandArgs& A, unsigned* own, const unsigned n) {
    unsigned w = own[n];
    if (w & kOwnPhantom) {
        bool held = false;
        for (int s = 0; s < kPhSlots; ++s) {
            const unsigned ph = A.phantom[(size_t)kPhSlots * n + s];
            if (!ph) continue;
            if (w & own_won_bit(s)) { A.phantom_leaf[ph] = -1; A.phantom[(size_t)kPhSlots * n + s] = 0u; }   // the holder owns it now (or lost it for good to a later thief)
            else held = true;
        }
        w &= ~kOwnWon;
        if (!held) w &= ~kOwnPhantom;
        own[n] = w;
    }
    const unsigned l = w & kOwnMask;
    if (l) A.list_raw[A.off[l] + atomicAdd(&A.fill[l], 1u)] = n;
    if (w & kOwnPhantom)
        for (int s = 0; s < kPhSlots; ++s) { const unsigned ph = A.phantom[(size_t)kPhSlots * n + s]; if (ph) A.list_raw[A.off[ph] + atomicAdd(&A.fill[ph], 1u)] = n; }
}

// one helper, one warp: leaves in idx order (ranks by counting), then SupervoxelHelper::updateCentroid -- the leaves' data are
// staged 32 at a time in shared memory, lanes 0..9 each run one ordered accumulator chain (n0..n3, x,y,z, r,g,b)
template <int ROW = 12>
__device__ __forceinline__ void expand_fold_helper(const ExpandArgs& A, const unsigned* cnt_final, const unsigned l, const int lane,
                                                   unsigned* s_sorted, float* stage) {
    const unsigned s = A.off[l], c = cnt_final[l];
    if (c == 0) { if (lane == 0 && A.rounds > 0) A.cen.xyz[l].w = 0.0f; return; }   // helper erased (no leaves)
    // ranks by counting (leaf sets are small; values are distinct)
    unsigned sorted_mine = 0u;
    for (unsigned ib = 0; ib < c; ib += 32) {
        const unsigned i = ib + lane;
        const unsigned v = i < c ? A.list_raw[s + i] : 0xffffffffu;
        unsigned rank = 0;
        for (unsigned jb = 0; jb < c; jb += 32) {
            const unsigned x = (c <= 32) ? v : (jb + lane < c ? A.list_raw[s + jb + lane] : 0xffffffffu);
            const unsigned m = min(32u, c - jb);
            for (unsigned t = 0; t < m; ++t) rank += __shfl_sync(kFull, x, t) < v ? 1u : 0u;
        }
        if (i < c) {
            A.list_sorted[s + rank] = v; A.pos_label[s + rank] = l;
            if (c <= 32) s_sorted[rank] = v;
        }
    }
    __syncwarp();
    if (A.rounds == 0) return;
    float acc = 0.0f;
    for (unsigned base = 0; base < c; base += 32) {
        const unsigned m = min(32u, c - base);
        if (base + lane < c) {
            sorted_mine = c <= 32 ? s_sorted[lane] : ldcg_u(A.list_sorted + s + base + lane);   // same-phase data: L2
            const float4 vn = A.vox_nrm[sorted_mine], vx = A.vox_xyz[sorted_mine], vc = A.vox_rgb[sorted_mine];
            float* row = stage + lane * ROW;
            row[0] = vn.x; row[1] = vn.y; row[2] = vn.z; row[3] = vn.w;
            row[4] = vx.x; row[5] = vx.y; row[6] = vx.z; row[7] = vc.x; row[8] = vc.y; row[9] = vc.z;
        }
        __syncwarp();
        if (lane < 10) for (unsigned j = 0; j < m; ++j) acc += stage[j * ROW + lane];
        __syncwarp();
    }
    float n0 = __shfl_sync(kFull, acc, 0), n1 = __shfl_sync(kFull, acc, 1), n2 = __shfl_sync(kFull, acc, 2), n3 = __shfl_sync(kFull, acc, 3);
    float x = __shfl_sync(kFull, acc, 4), y = __shfl_sync(kFull, acc, 5), z = __shfl_sync(kFull, acc, 6);
    float r = __shfl_sync(kFull, acc, 7), g = __shfl_sync(kFull, acc, 8), b = __shfl_sync(kFull, acc, 9);
    if (lane == 0) {
        float zz = sum4(n0 * n0, n1 * n1, n2 * n2, n3 * n3);
        if (zz > 0.0f) { float sq = sqrtf(zz); n0 /= sq; n1 /= sq; n2 /= sq; n3 /= sq; }
        const float cf = (float)c;
        A.cen.nrm[l] = make_float4(n0, n1, n2, n3);
        A.cen.xyz[l] = make_float4(x / cf, y / cf, z / cf, cf);
        A.cen.rgb[l] = make_float4(r / cf, g / cf, b / cf, 0.0f);
    }
    __syncwarp();
}

// surviving helpers in label order (makeSupervoxels): exclusive scan of (count > 0) by ONE block
__device__ __forceinline__ void expand_alive_scan(const ExpandArgs& A, const unsigned* cnt_final, unsigned* s_warp, unsigned* s_carry) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) { (*s_carry) = 0; A.ctl->n_pos = ldcg_u(&A.ctl->cursor); }
    __syncthreads();
    for (unsigned base = 1; base <= A.S0; base += blockDim.x) {      // alive ranks: exclusive scan of (count > 0)
        const unsigned l = base + threadIdx.x;
        const unsigned a = (l <= A.S0 && ldcg_u(cnt_final + l) > 0u) ? 1u : 0u;
        unsigned v = a;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { unsigned t = __shfl_up_sync(kFull, v, o); if (lane >= o) v += t; }
        if (lane == 31) s_warp[warp] = v;
        __syncthreads();
        unsigned wb = 0;
        for (int w = 0; w < warp; ++w) wb += s_warp[w];
        const unsigned carry = (*s_carry);
        if (a) { const unsigned rank = carry + wb + v - 1u; A.sv_label[rank] = l; A.rank_of_label[l] = rank; }
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) (*s_carry) = carry + wb + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) A.ctl->n_sv = (*s_carry);
}

// shared memory of one CTA (declared by the kernels: static __shared__ inside a function template is shared between its
// instantiations by nvcc 12.9, which broke the 512-thread instantiation)
template <int THREADS>
struct ExpandSmem {
    static constexpr int ROW = THREADS > 512 ? 10 : 12;       // floats per staged leaf (10 used); 1024 threads must stay within 48 KB static
    unsigned s_warp[32];
    unsigned s_carry;
    unsigned s_sorted[THREADS / 32][32];
    float s_stage[THREADS / 32][32][ROW];
};

template <int THREADS, bool CLUSTER>
__device__ __forceinline__ void expand_body(const ExpandArgs& A, ExpandSmem<THREADS>& SM, const unsigned cta, const unsigned nblocks) {   // cta of nblocks CTAs work on this frame
    constexpr int ROW = ExpandSmem<THREADS>::ROW;
    unsigned (&s_warp)[32] = SM.s_warp;
    unsigned& s_carry = SM.s_carry;
    auto& s_sorted = SM.s_sorted;
    auto& s_stage = SM.s_stage;
    const unsigned tid = cta * blockDim.x + threadIdx.x, nthreads = nblocks * blockDim.x;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const unsigned gwarp = tid >> 5, nwarps = nthreads >> 5;
    const unsigned V = A.V, S0 = A.S0;
    ExpandCtl* ctl = A.ctl;
    unsigned phase = 0;
    unsigned long long t_prev = globaltimer_ns();

    // ---- createSupervoxelHelpers -------------------------------------------------------------------
    for (unsigned v = tid; v < V; v += nthreads) { A.owner[0][v] = 0u; A.dist[0][v] = FLT_MAX; A.st[0][v] = kNoSteal; for (int s = 0; s < kPhSlots; ++s) A.phantom[(size_t)kPhSlots * v + s] = 0u; }
    for (unsigned l = tid; l < S0 + 2; l += nthreads) {
        if (!A.keep_centroids) {
            A.cen.xyz[l] = make_float4(0, 0, 0, l >= 1 && l <= S0 ? 1.0f : 0.0f);   // SupervoxelHelper::centroid_ starts at zero (literal)
            A.cen.rgb[l] = make_float4(0, 0, 0, 0); A.cen.nrm[l] = make_float4(0, 0, 0, 0);
        }
        A.phantom_leaf[l] = -1; A.count[0][l] = 0u; A.count[1][l] = 0u; A.off[l] = 0u;
    }
    expand_barrier<CLUSTER>(ctl, nblocks, phase);
    for (unsigned i = tid; i < S0; i += nthreads) if (A.seeds[i] >= 0) atomicMax(&A.owner[0][A.seeds[i]], i + 1u);      // addLeaf: the last helper owns
    expand_barrier<CLUSTER>(ctl, nblocks, phase);
    for (unsigned i = tid; i < S0; i += nthreads) {
        if (A.seeds[i] < 0) continue;
        const unsigned u = (unsigned)A.seeds[i];
        if ((ldcg_u(A.owner[0] + u) & kOwnMask) == i + 1u) continue;
        bool placed = false;
        for (int s = 0; s < kPhSlots && !placed; ++s) placed = atomicCAS(&A.phantom[(size_t)kPhSlots * u + s], 0u, i + 1u) == 0u;
        if (!placed) atomicOr(&ctl->error, (unsigned)EXPAND_ERR_TRIPLE);        // more than kPhSlots + 1 seed cells on one voxel: not modelled
        A.phantom_leaf[i + 1] = (int)u;
        atomicOr(&A.owner[0][u], kOwnPhantom);
    }
    expand_barrier<CLUSTER>(ctl, nblocks, phase);
    XPHASE(0);

    int cur = 0;
    unsigned k = 0;                                             // running sweep number: parity selects the steal-table / count buffers
    const int n_rounds = A.rounds > 0 ? A.rounds : 1;           // rounds == 0: helpers keep their seed leaf, lists only
    for (int round = 0; round < n_rounds; ++round) {
        unsigned* cnt_final = A.count[0];
        if (A.rounds > 0) {
            // ---- expand(): sweeps to the fixed point of the steal table; every sweep also tallies the helper sizes
            // its result implies, so the confirming sweep leaves the round's counts behind --------------------------
            bool converged = false;
            for (int s = 0; s < kExpandMaxSweeps && !converged; ++s, ++k) {
                const unsigned* own0 = A.owner[cur]; const float* dst0 = A.dist[cur];
                unsigned* own1 = A.owner[cur ^ 1]; float* dst1 = A.dist[cur ^ 1];
                const unsigned* st_in = A.st[k & 1]; unsigned* st_out = A.st[(k + 1) & 1];
                unsigned* cnt = A.count[k & 1]; unsigned* cnt_next = A.count[(k + 1) & 1];
                unsigned any_change = 0;
                for (unsigned l = tid; l < S0 + 2; l += nthreads) cnt_next[l] = 0u;
                if (tid == 0) { ctl->changed[(k + 2u) & 63u] = 0u; ctl->cursor = 0u; }
                const unsigned char* chg_in = s > 0 ? A.chg[k & 1] : nullptr;     // the first sweep of a round evaluates everything
                unsigned char* chg_out = A.chg[(k + 1) & 1];
                for (unsigned n = tid; n < V; n += nthreads) expand_sweep_voxel(A, n, own0, dst0, own1, dst1, st_in, st_out, cnt, any_change, chg_in, chg_out);
                if (__syncthreads_or(any_change) && threadIdx.x == 0) atomicOr(&ctl->changed[k & 63u], 1u);
                expand_barrier<CLUSTER>(ctl, nblocks, phase);
                converged = ldcg_u(&ctl->changed[k & 63u]) == 0u;
                cnt_final = cnt;
                if (tid == 0) atomicAdd(&ctl->sweeps_total, 1u);
            }
            if (!converged && tid == 0) atomicOr(&ctl->error, (unsigned)EXPAND_ERR_SWEEPS);
            cur ^= 1;
            XPHASE(1);
        } else {
            // no expansion rounds: sizes straight from createSupervoxelHelpers
            const unsigned* own = A.owner[cur];
            for (unsigned n = tid; n < V; n += nthreads) {
                const unsigned w = ldcg_u(own + n);
                if (w & kOwnMask) atomicAdd(&cnt_final[w & kOwnMask], 1u);
                if (w & kOwnPhantom) for (int s = 0; s < kPhSlots; ++s) { const unsigned h = ldcg_u(A.phantom + (size_t)kPhSlots * n + s); if (h) atomicAdd(&cnt_final[h], 1u); }
            }
            expand_barrier<CLUSTER>(ctl, nblocks, phase);
            XPHASE(2);
        }
        // ---- alloc: one contiguous leaf list per helper (warp-aggregated bump allocation; helper order is irrelevant) ----
        for (unsigned base = gwarp * 32u; base < S0; base += nwarps * 32u) expand_alloc_warp(A, cnt_final, base, lane);
        expand_barrier<CLUSTER>(ctl, nblocks, phase);
        XPHASE(3);
        // ---- fill: commit the round (a phantom leaf its holder stole becomes a regular leaf), unordered member lists ----
        {
            unsigned* own = A.owner[cur];
            unsigned* st_next = A.st[k & 1];
            for (unsigned n = tid; n < V; n += nthreads) {
                expand_fill_voxel(A, own, n);
                st_next[n] = kNoSteal;
            }
        }
        expand_barrier<CLUSTER>(ctl, nblocks, phase);
        XPHASE(4);
        // ---- per helper (one warp): leaves in idx order, then SupervoxelHelper::updateCentroid: the leaves' data are
        // staged 32 at a time in shared memory, lanes 0..9 each run one ordered accumulator chain (n0..n3, x,y,z, r,g,b) ----
        {
            float* stage = &s_stage[wib][0][0];
            for (unsigned l = 1 + gwarp; l <= S0; l += nwarps) {
                expand_fold_helper<ROW>(A, cnt_final, l, lane, &s_sorted[wib][0], stage);
            }
        }
        expand_barrier<CLUSTER>(ctl, nblocks, phase);
        XPHASE(5);
        // ---- after the last round: clean labels, per-helper bounds, surviving helpers in label order (makeSupervoxels) ----
        if (round == n_rounds - 1) {
            const unsigned* own = A.owner[cur]; const float* dst = A.dist[cur];
            for (unsigned n = tid; n < V; n += nthreads) { A.labels_out[n] = ldcg_u(own + n) & kOwnMask; A.dist_out[n] = ldcg_f(dst + n); }
            for (unsigned l = tid; l < S0 + 2; l += nthreads) A.seg_end[l] = (l >= 1 && l <= S0) ? ldcg_u(A.off + l) + ldcg_u(cnt_final + l) : 0u;
            if (cta == 0) {
                expand_alive_scan(A, cnt_final, s_warp, &s_carry);
            }
            XPHASE(6);
        }
    }
}

// cooperative grid over the whole GPU (any V): software grid barrier through L2
__global__ void __launch_bounds__(kExpandThreads, F3PS_EXPAND_MIN_BLOCKS) expand_persistent_kernel(ExpandArgs A) {
    __shared__ ExpandSmem<kExpandThreads> SM;
    expand_body<kExpandThreads, false>(A, SM, blockIdx.x, gridDim.x);
}

// ONE thread-block cluster per frame (up to 16 CTAs of 1024 threads, launched with clusterDim == gridDim): the phases meet at
// the hardware cluster barrier.  A VGA frame (34 k voxels, ~110 barriers) is bound by the meeting points, not by the work
// between them; a cluster also leaves the other SMs to the frames next to it in a sweep (no cooperative launch, which the
// driver runs one at a time).
constexpr int kExpandClusterThreads = 1024;
constexpr int kExpandClusterMax = 16;
__global__ void __launch_bounds__(kExpandClusterThreads, 1) expand_cluster_kernel(ExpandArgs A) {
    __shared__ ExpandSmem<kExpandClusterThreads> SM;
    expand_body<kExpandClusterThreads, true>(A, SM, blockIdx.x, gridDim.x);
}

} // namespace f3ps
