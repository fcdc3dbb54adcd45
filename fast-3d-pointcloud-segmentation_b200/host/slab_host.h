// slab_host.h -- slab mode driven from C++ over NCCL: ONE very large cloud on several GPUs (SURVEY.md section 8e row 2,
// BASELINE config 5).  The reference runs pcl::SupervoxelClustering::extract + Clustering::cluster on the whole cloud in one
// thread (/root/reference/src/supervoxel_clustering.cpp:348-367, 408-449); here every rank (one host thread + one CUDA stream +
// one f3ps handle per GPU, one ncclComm_t each) starts with an arbitrary share of the points and the cloud is cut into
// contiguous ranges of the x-major Morton key -- PCL's leaf order -- so every ordered float sum keeps its order and the result is
// bit-identical to one handle processing the whole cloud.  Same protocol as f3ps/slab.py (torch.distributed), same per-rank C-ABI
// pieces (include/f3ps.h: f3ps_slab_*, splitter choice and voxel-table assembly included); this driver adds only the exchanges,
// NCCL collectives issued on the handle's stream.
#pragma once
#include <cstdint>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "f3ps.h"

namespace f3ps_host {

struct SlabParams {
    float voxel_res = 0.008f, seed_res = 0.08f, color_imp = 0.2f, spatial_imp = 0.4f, normal_imp = 1.0f;
    int use_transform = 1, fold_negative_z = 1;
    int color_distance = 0, geometric_distance = 0, merging = 0;
    float lambda = 0.5f;
    int bins = 500;
    float threshold = 0.2f;
    bool merge = true;
};

// one rank's share of the cloud: host memory, or (on_device) memory of that rank's GPU -- the scans it recorded, already in HBM
struct SlabShare { const void* points = nullptr; int64_t n = 0; int stride = 32; bool on_device = false; };

struct SlabInfo {                     // per rank, after run()
    int64_t n_local = 0, n_received = 0, v_local = 0, V = 0, own_lo = 0, own_hi = 0;
    int sweeps = 0;
    uint64_t bytes_exchanged = 0;
    std::vector<std::pair<std::string, float>> stage_ms;   // in stage order; the last entry is "total"
    std::string error;                // empty = ok
};

class SlabRun {
public:
    explicit SlabRun(const std::vector<int>& devices);      // one rank per listed CUDA device (ncclCommInitAll)
    ~SlabRun();
    SlabRun(const SlabRun&) = delete;
    SlabRun& operator=(const SlabRun&) = delete;
    int world() const { return (int)devices_.size(); }
    bool ok() const { return init_error_.empty(); }
    const std::string& init_error() const { return init_error_; }
    // Runs the whole path; shares[r] = rank r's points (the global input order is the concatenation in rank order).
    // Afterwards EVERY rank's handle holds the complete result (K7 is replayed by every rank).  Returns 0, or the first failing
    // rank's f3ps status (info(r).error says what).
    int run(const std::vector<SlabShare>& shares, const SlabParams& p);
    f3ps_ctx* handle(int rank) const { return ctx_[(size_t)rank]; }
    const SlabInfo& info(int rank) const { return info_[(size_t)rank]; }

private:
    void rank_main(int rank, const SlabShare& share, const SlabParams& p);
    std::vector<int> devices_;
    std::vector<f3ps_ctx*> ctx_;
    std::vector<void*> stream_;       // cudaStream_t
    std::vector<void*> comm_;         // ncclComm_t
    std::vector<std::shared_ptr<void>> mem_;   // per rank: the exchange buffers, kept from run to run
    std::vector<SlabInfo> info_;
    std::vector<int> status_;
    std::string init_error_;
};

}  // namespace f3ps_host
