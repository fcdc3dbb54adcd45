// context.cuh -- the handle behind f3ps_ctx: device buffers, device-resident scalars, launch helpers.
#pragma once
#include <string>
#include <vector>
#include "../../include/f3ps.h"
#include "common.cuh"
#include "radix_sort.cuh"
#include "kernels_vccs.cuh"
#include "kernels_expand.cuh"
#include "kernels_slab.cuh"
#include "kernels_graph.cuh"
#include "kernels_merge.cuh"
#include "kernels_merge_lean.cuh"
#include "kernels_eval.cuh"
#include "kernels_segments.cuh"

namespace f3ps {

// Owning device buffer: freed by its destructor, so a handle's `delete` releases every buffer it ever grew
// (f3ps_destroy used to walk an explicit list that missed the threshold-sweep and slab buffers).
struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap && p) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// the members of every segment of one level, grouped (f3ps_get_segment_points / _voxels): sort buffers, offsets[K+1] and the
// partial offsets (kernels_segments.cuh), and where the grouped indices ended up; level -1 = nothing grouped since the last merge
struct SegCsr {
    DevBuf keys_a, keys_b, vals_a, vals_b, offsets, counts;
    const unsigned* index = nullptr;
    int level = -1; unsigned n = 0, K = 0;
    long long* off() const { return offsets.as<long long>(); }
    unsigned* chunk_off() const { return reinterpret_cast<unsigned*>(offsets.as<long long>() + K + 1); }
};

// everything the kernels count or decide lives here, on the device; the host mirrors it on demand
struct DevScalars {
    FrameParams fp;
    unsigned n_valid, n_voxels, n_cells, n_seeds;
    unsigned pad_sv, n_edges, n_out, edge_overflow;
    unsigned bad_bin, nan_weights_init, pad0, pad1;
    float lambda; float padf[3];
    ExpandCtl xctl;
    MergeCtl mctl;
    SeedBox sb;
};

enum Progress { P_NONE = 0, P_INPUT, P_VOXELS, P_NEIGHBORS, P_NORMALS, P_SEEDS, P_EXPANDED, P_GRAPH, P_MERGED };

} // namespace f3ps

struct f3ps_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t private_stream = nullptr;   // created by the handle (f3ps_create without a stream); destroyed with it
    std::string err;
    f3ps::VccsParams vp{0.008f, 0.08f, 0.2f, 0.4f, 1.0f, 1, 1};
    f3ps::MergeParams mp{0, 0, 1, 0.5f, 500};
    int progress = f3ps::P_NONE;
    bool graph_from_host = false;
    long long launches = 0;

    // input
    const uint8_t* d_points = nullptr; int64_t n_points = 0; int stride = 32;
    f3ps::DevBuf in_buf;
    // scalars
    f3ps::DevScalars* d_sc = nullptr;
    f3ps::DevScalars* h_sc = nullptr;      // pinned mirror
    short* d_lab_lut = nullptr;
    // host-known sizes (after the syncs)
    int depth = 0; unsigned V = 0, n_valid = 0, n_cells = 0, S0 = 0, S = 0, E = 0, n_out = 0;
    int rounds = 0, key_bits = 0;
    bool key64 = false;

    // K1
    f3ps::DevBuf keys_a, keys_b, vals_a, vals_b, starts, point_voxel, sort_scratch, compact_scratch;
    void* sorted_keys = nullptr; unsigned* sorted_idx = nullptr;
    f3ps::DevBuf vox_xyz, vox_rgb, vox_key;
    // K2
    f3ps::DevBuf hash_slots, hash_vals, nbr_row, nbr_col;
    unsigned hash_mask = 0;
    // K3
    f3ps::DevBuf vox_normal, vox_curv;
    // K4
    f3ps::DevBuf cell_code, cell_code_b, cell_vox, cell_vox_b, vox_cell, cell_start, cell_codes, cell_nn, cell_keep, seeds;
    f3ps::DevBuf lean_big;                    // K7 resident kernel, BIG variant: per-edge / per-region tables + set-up scratch in global memory
    f3ps::DevBuf seeds_refine;                // reseedSupervoxels: one voxel per helper, -1 = erased (f3ps_refine)
    // K5
    f3ps::DevBuf owner0, dist0;                       // results: clean label / stored distance per voxel
    f3ps::DevBuf chg_a, chg_b;                        // active-set flags of the sweeps
    f3ps::DevBuf own_a, own_b, dst_a, dst_b, st0, st1, phantom, phantom_leaf, lab_count, lab_count2, lab_fill;
    f3ps::DevBuf cen_xyz, cen_rgb, cen_nrm, lab_keys_a, lab_keys_b, lab_vals_a, lab_vals_b, seg_start, seg_end;
    int expand_blocks_per_sm = 0, sm_count = 0;
    int expand_ctas = 0;                // > 0: cap of K5's cooperative grid (f3ps_set_expand_sharing)
    unsigned* sorted_label = nullptr; unsigned* sorted_vox = nullptr;
    // K6
    f3ps::DevBuf sv_label, rank_of_label, run_start, run_end, pos_run, edge_set, edge_keys_a, edge_keys_b, edge_vals_a, edge_vals_b;
    f3ps::DevBuf dbits_a, dbits_b, dbits_c, dbits_d, cdf_c, cdf_g, cdf_hist;
    f3ps::DevBuf reg_init, reg_work, edge_init, edge_work;     // packed RegionArrays / EdgeArrays storage
    f3ps::RegionArrays R0{}, R1{}; f3ps::EdgeArrays E0{}, E1{};
    unsigned long long* sorted_edge_keys = nullptr;
    unsigned edge_set_mask = 0; int edge_kb = 0;
    // K7
    f3ps::DevBuf mlog, run_out_off, run_dense, region_dense, out_xyz, out_label, out_voxel, vox_segment;
    f3ps::DevBuf pos_data_buf, merge_scratch, adj_pool, merge_trace;
    unsigned merge_trace_first = 0;
    const float4* pos_data = nullptr;   // voxel (x,y,z,rgba) in position order (what the merge folds stream)
    int merge_path = 0;                 // what the last replay ran (f3ps_counts.merge_path)
    int merge_kernel_choice = 0;        // 0 auto, 2 general, 3 resident with its tables in L2, 4 = auto with phase counters in the shared-memory variant, 5 = 3 with phase counters
    f3ps::MergeLog ML{};
    unsigned n_pos = 0;           // positions of the label-ordered voxel list
    const unsigned* order = nullptr;
    const float4* gxyz = nullptr; // voxel xyz(+rgba) array the graph stages read

    static constexpr int kEvents = 11;   // 0..8 stage boundaries, 9/10 around the merge kernel alone
    cudaEvent_t ev[kEvents] = {};
    bool ev_valid[kEvents] = {};
    cudaEvent_t ev_batch = nullptr;    // f3ps_merge_batch: set-up done
    // f3ps_merge_batch, as the lead of a chunk: the DevScalars of the chunk's frames, gathered on the device and their pinned mirror
    f3ps::DevBuf batch_sc;
    f3ps::DevScalars* h_batch_sc = nullptr;
    cudaEvent_t ev_wait = nullptr;     // blocking-sync event for sweeps (f3ps_set_blocking_wait)
    bool blocking_wait = false;
    // slab mode (f3ps_slab_*): injected global frame, histogram binning of f3ps_slab_keys (bin = key >> slab_shift,
    // 1 << slab_bits bins; 0 bits: keys have not run), owned voxel range
    bool slab_frame = false; f3ps::FrameParams slab_fp{};
    int slab_bits = 0, slab_shift = 0;
    bool slab_range = false; unsigned own_begin = 0, own_end = 0;
    f3ps::DevBuf slab_dest, slab_tot, slab_spare;   // slab_spare: this rank's voxel slice while f3ps_slab_set_voxels moves it
    f3ps::DevBuf ev_dense, ev_truth, ev_table;   // f3ps_eval_thresholds, f3ps_eval_label_pairs
    // segmentation levels (f3ps_merge_levels; every merge records its own threshold as the one level).  The tables are built on
    // the first getter call after the merge: forest, per-level merge counts and per-supervoxel labels, then the voxel table.
    std::vector<float> lv_thr;          // thresholds of the recorded levels; empty: no merged state to read levels from
    unsigned lv_M = 0;                  // merges of the replay the levels are prefixes of
    int lv_built = 0;                   // 0 nothing, 1 level tables of lv_thr, 2 and the voxel table
    std::vector<int32_t> lv_m_h, lv_nseg_h;
    f3ps::DevBuf lv_small, lv_parent, lv_when, lv_dense, lv_seg, lv_vox, lv_points;
    // segment extraction: the point and the voxel grouping of the last level asked for, kept until the next merge
    f3ps::SegCsr seg_points, seg_voxels;
    f3ps::DevBuf seg_part, seg_info;
    f3ps::DevBuf graph_vox;             // f3ps_set_graph: voxel index as passed in, per position
    int expand_kernel_choice = 0;       // f3ps_set_expand_kernel: 0 auto, 1 cooperative grid, 2 one cluster
    int expand_cluster_ctas = 0;        // cap of the cluster size (0 = by V, at most 16)
    bool expand_cluster_attr_set = false;
    bool lambda_attr_set = false;
};
