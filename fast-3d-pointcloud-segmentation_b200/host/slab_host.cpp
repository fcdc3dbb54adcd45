// slab_host.cpp -- see slab_host.h.  One host thread per GPU; every exchange is an NCCL collective on the rank's stream, so it
// orders against the f3ps kernels without extra events.  The protocol follows f3ps/slab.py step by step (the Python driver stays
// for the torch.distributed / gloo tests); stage names and the exchanged-byte count are the same.  The splitter rule and the
// assembly of the replicated voxel table are library calls, so both drivers cut a cloud in the same place by construction.
#include "slab_host.h"

#include <cuda_runtime.h>
#include <nccl.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <stdexcept>
#include <thread>

namespace f3ps_host {

namespace {
constexpr int kTopBits = 12;

struct Fail : std::runtime_error { int code; Fail(int c, const std::string& m) : std::runtime_error(m), code(c) {} };
void cu(cudaError_t e, const char* what) { if (e != cudaSuccess) throw Fail(F3PS_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e)); }
void nc(ncclResult_t r, const char* what) { if (r != ncclSuccess) throw Fail(F3PS_ERR_CUDA, std::string(what) + ": " + ncclGetErrorString(r)); }

struct DevMem {                                    // cudaMalloc'ed buffer of one rank (grows, never shrinks)
    void* p = nullptr; size_t cap = 0;
    ~DevMem() { if (p) cudaFree(p); }
    void* ensure(size_t bytes) {
        if (bytes > cap) { if (p) cudaFree(p); p = nullptr; cu(cudaMalloc(&p, std::max<size_t>(bytes, 256)), "cudaMalloc"); cap = std::max<size_t>(bytes, 256); }
        return p;
    }
};
struct RankMem { int device = 0; DevMem small, send, recv; };   // exchange buffers of one rank, reused by every run
}  // namespace

SlabRun::SlabRun(const std::vector<int>& devices) : devices_(devices) {
    const size_t w = devices_.size();
    ctx_.assign(w, nullptr); stream_.assign(w, nullptr); comm_.assign(w, nullptr); info_.resize(w); status_.assign(w, 0);
    try {
        if (w == 0) throw Fail(F3PS_ERR_INVALID_ARGUMENT, "no devices");
        std::vector<ncclComm_t> comms(w);
        nc(ncclCommInitAll(comms.data(), (int)w, devices_.data()), "ncclCommInitAll");
        for (size_t r = 0; r < w; ++r) comm_[r] = comms[r];
        for (size_t r = 0; r < w; ++r) {
            cu(cudaSetDevice(devices_[r]), "cudaSetDevice");
            cudaStream_t s;
            cu(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking), "cudaStreamCreate");
            stream_[r] = s;
            const int rc = f3ps_create(devices_[r], s, &ctx_[r]);
            if (rc) throw Fail(rc, "f3ps_create failed on device " + std::to_string(devices_[r]));
            const int dev = devices_[r];
            mem_.push_back(std::shared_ptr<void>(new RankMem{dev}, [](void* p) { RankMem* m = (RankMem*)p; cudaSetDevice(m->device); delete m; }));
        }
    } catch (const Fail& f) { init_error_ = f.what(); }
}

SlabRun::~SlabRun() {
    for (size_t r = 0; r < devices_.size(); ++r) {
        cudaSetDevice(devices_[r]);
        if (ctx_[r]) f3ps_destroy(ctx_[r]);
        if (comm_[r]) ncclCommDestroy((ncclComm_t)comm_[r]);
        if (stream_[r]) cudaStreamDestroy((cudaStream_t)stream_[r]);
    }
}

int SlabRun::run(const std::vector<SlabShare>& shares, const SlabParams& p) {
    if (!ok() || (int)shares.size() != world()) return F3PS_ERR_INVALID_ARGUMENT;
    std::vector<std::thread> th;
    for (int r = 0; r < world(); ++r) th.emplace_back([this, r, &shares, &p] { rank_main(r, shares[(size_t)r], p); });
    for (auto& t : th) t.join();
    for (int r = 0; r < world(); ++r) if (status_[(size_t)r]) return status_[(size_t)r];
    return F3PS_OK;
}

void SlabRun::rank_main(int rank, const SlabShare& share, const SlabParams& p) {
    SlabInfo& info = info_[(size_t)rank];
    info = SlabInfo();
    status_[(size_t)rank] = 0;
    const int world = this->world();
    f3ps_ctx* ctx = ctx_[(size_t)rank];
    cudaStream_t st = (cudaStream_t)stream_[(size_t)rank];
    ncclComm_t comm = (ncclComm_t)comm_[(size_t)rank];
    std::vector<std::pair<std::string, cudaEvent_t>> ev;
    try {
        cu(cudaSetDevice(devices_[(size_t)rank]), "cudaSetDevice");
        auto ok = [&](int rc, const char* what) { if (rc) throw Fail(rc, std::string(what) + ": " + f3ps_last_error(ctx)); };
        auto tick = [&](const char* name) { cudaEvent_t e; cu(cudaEventCreate(&e), "cudaEventCreate"); cu(cudaEventRecord(e, st), "cudaEventRecord"); ev.emplace_back(name, e); };
        uint64_t moved = 0;
        // ---- the collectives of the protocol ----
        auto all_reduce = [&](void* d, size_t count, ncclDataType_t t, ncclRedOp_t op, size_t elem) {
            if (world == 1 || count == 0) return;
            nc(ncclAllReduce(d, d, count, t, op, comm, st), "ncclAllReduce"); moved += count * elem;
        };
        // rows [b[r], b[r+1]) of `full` (elem bytes each) are valid on rank r; afterwards all rows are valid everywhere
        auto gather_slices = [&](void* full, const std::vector<int64_t>& b, size_t elem) {
            if (world == 1) return;
            nc(ncclGroupStart(), "ncclGroupStart");
            for (int r = 0; r < world; ++r) {
                const int64_t lo = b[(size_t)r], hi = b[(size_t)r + 1];
                if (hi <= lo) continue;
                char* part = (char*)full + (size_t)lo * elem;
                nc(ncclBroadcast(part, part, (size_t)(hi - lo) * elem, ncclChar, r, comm, st), "ncclBroadcast");
                moved += (uint64_t)(hi - lo) * elem;
            }
            nc(ncclGroupEnd(), "ncclGroupEnd");
        };
        auto slab_array = [&](int which, void*& ptr, int64_t& n, int& eb) { ok(f3ps_slab_array(ctx, which, &ptr, &n, &eb), "f3ps_slab_array"); };
        RankMem& M = *(RankMem*)mem_[(size_t)rank].get();
        DevMem &small = M.small, &send = M.send, &recv = M.recv;

        ok(f3ps_set_vccs_params(ctx, p.voxel_res, p.seed_res, p.color_imp, p.spatial_imp, p.normal_imp, p.use_transform, p.fold_negative_z), "f3ps_set_vccs_params");
        ok(f3ps_set_merge_params(ctx, p.color_distance, p.geometric_distance, p.merging, p.lambda, p.bins), "f3ps_set_merge_params");
        tick("start");
        ok(f3ps_slab_reset(ctx), "f3ps_slab_reset");
        const int64_t n_local = share.n;
        info.n_local = n_local;
        ok(f3ps_set_input(ctx, share.points, n_local, share.stride, share.on_device ? 1 : 0), "f3ps_set_input");
        // ---- K1a: the frame of the whole cloud (order-preserving encoded box: MIN of 3 words, MAX of 4) ----
        uint32_t* d_small = (uint32_t*)small.ensure(((size_t)8 + ((size_t)1 << kTopBits)) * 4 + (size_t)world * (size_t)world * 8 + 64);
        uint32_t* d_box = d_small;
        uint32_t* d_hist = d_small + 8;
        int64_t* d_mat = (int64_t*)(d_hist + ((size_t)1 << kTopBits));
        cu(cudaMemsetAsync(d_box, 0, 32, st), "memset");
        ok(f3ps_slab_bbox(ctx, d_box), "f3ps_slab_bbox");
        all_reduce(d_box, 3, ncclUint32, ncclMin, 4);
        all_reduce(d_box + 3, 4, ncclUint32, ncclMax, 4);
        ok(f3ps_slab_set_frame(ctx, d_box), "f3ps_slab_set_frame");
        // ---- K1b: keys, splitters, routing ----
        cu(cudaMemsetAsync(d_hist, 0, ((size_t)4) << kTopBits, st), "memset");
        ok(f3ps_slab_keys(ctx, kTopBits, d_hist), "f3ps_slab_keys");
        all_reduce(d_hist, (size_t)1 << kTopBits, ncclUint32, ncclSum, 4);
        void* d_send = send.ensure((size_t)std::max<int64_t>(1, n_local) * 16);
        std::vector<int64_t> send_counts((size_t)world, 0);
        ok(f3ps_slab_route(ctx, world, d_hist, d_send, send_counts.data()), "f3ps_slab_route");
        tick("route");
        // count matrix [src][dst] (all-gather of the rows), then the points to the rank owning their key range
        std::vector<int64_t> mat((size_t)world * (size_t)world, 0);
        if (world > 1) {
            cu(cudaMemcpyAsync(d_mat + (size_t)rank * (size_t)world, send_counts.data(), (size_t)world * 8, cudaMemcpyHostToDevice, st), "memcpy counts");
            nc(ncclAllGather(d_mat + (size_t)rank * (size_t)world, d_mat, (size_t)world, ncclInt64, comm, st), "ncclAllGather");
            cu(cudaMemcpyAsync(mat.data(), d_mat, mat.size() * 8, cudaMemcpyDeviceToHost, st), "memcpy matrix");
            cu(cudaStreamSynchronize(st), "sync");
        } else mat[0] = send_counts[0];
        std::vector<int64_t> recv_counts((size_t)world), soff((size_t)world + 1, 0), roff((size_t)world + 1, 0);
        for (int r = 0; r < world; ++r) {
            recv_counts[(size_t)r] = mat[(size_t)r * (size_t)world + (size_t)rank];
            soff[(size_t)r + 1] = soff[(size_t)r] + send_counts[(size_t)r]; roff[(size_t)r + 1] = roff[(size_t)r] + recv_counts[(size_t)r];
        }
        const int64_t n_recv = roff[(size_t)world];
        info.n_received = n_recv;
        void* d_recv = recv.ensure((size_t)std::max<int64_t>(1, n_recv) * 16);
        if (world == 1) cu(cudaMemcpyAsync(d_recv, d_send, (size_t)n_recv * 16, cudaMemcpyDeviceToDevice, st), "memcpy points");
        else {
            nc(ncclGroupStart(), "ncclGroupStart");
            for (int r = 0; r < world; ++r) {
                if (send_counts[(size_t)r]) nc(ncclSend((char*)d_send + (size_t)soff[(size_t)r] * 16, (size_t)send_counts[(size_t)r] * 16, ncclChar, r, comm, st), "ncclSend");
                if (recv_counts[(size_t)r]) nc(ncclRecv((char*)d_recv + (size_t)roff[(size_t)r] * 16, (size_t)recv_counts[(size_t)r] * 16, ncclChar, r, comm, st), "ncclRecv");
            }
            nc(ncclGroupEnd(), "ncclGroupEnd");
            moved += (uint64_t)soff[(size_t)world] * 16;
        }
        tick("all_to_all");
        // ---- K1c: voxels of the owned slab, then the replicated table ----
        ok(f3ps_set_input(ctx, d_recv, n_recv, 16, n_recv ? 1 : 0), "f3ps_set_input(received)");
        ok(f3ps_voxelize(ctx), "f3ps_voxelize");
        f3ps_counts c;
        ok(f3ps_get_counts(ctx, &c), "f3ps_get_counts");
        const int64_t v_local = c.n_voxels;
        info.v_local = v_local;
        std::vector<int64_t> vb((size_t)world + 1, 0);
        if (world > 1) {
            cu(cudaMemcpyAsync(d_mat + rank, &v_local, 8, cudaMemcpyHostToDevice, st), "memcpy v_local");
            nc(ncclAllGather(d_mat + rank, d_mat, 1, ncclInt64, comm, st), "ncclAllGather");
            std::vector<int64_t> vl((size_t)world);
            cu(cudaMemcpyAsync(vl.data(), d_mat, (size_t)world * 8, cudaMemcpyDeviceToHost, st), "memcpy v");
            cu(cudaStreamSynchronize(st), "sync");
            for (int r = 0; r < world; ++r) vb[(size_t)r + 1] = vb[(size_t)r] + vl[(size_t)r];
        } else vb[1] = v_local;
        const int64_t V = vb[(size_t)world], lo = vb[(size_t)rank], hi = vb[(size_t)rank + 1];
        info.V = V; info.own_lo = lo; info.own_hi = hi;
        ok(f3ps_slab_set_voxels(ctx, V, lo), "f3ps_slab_set_voxels");
        tick("voxelize");
        if (V) {
            void* ptr; int64_t n; int eb;
            for (int which : {F3PS_SLAB_VOX_XYZ, F3PS_SLAB_VOX_RGB, F3PS_SLAB_VOX_KEY}) { slab_array(which, ptr, n, eb); gather_slices(ptr, vb, (size_t)eb); }
        }
        tick("gather_voxels");
        // ---- K2 (replicated), K3 (owned slice + exchange), K4 (replicated) ----
        ok(f3ps_neighbors(ctx), "f3ps_neighbors");
        tick("neighbors");
        ok(f3ps_normals(ctx), "f3ps_normals");
        if (V) {
            void* ptr; int64_t n; int eb;
            slab_array(F3PS_SLAB_VOX_NORMAL, ptr, n, eb); gather_slices(ptr, vb, (size_t)eb);
            slab_array(F3PS_SLAB_VOX_CURV, ptr, n, eb); gather_slices(ptr, vb, (size_t)eb);
        }
        tick("normals");
        ok(f3ps_seeds(ctx), "f3ps_seeds");
        tick("seeds");
        // ---- K5 on the replicated table: the kernel of one handle, no exchange ----
        ok(f3ps_expand(ctx), "f3ps_expand");
        ok(f3ps_get_counts(ctx, &c), "f3ps_get_counts");
        info.sweeps = c.sweeps;
        tick("expand");
        // ---- K6, K7 on the replicated tables: K7 does not shard ("replicas only"), every rank replays it ----
        ok(f3ps_graph(ctx), "f3ps_graph");
        tick("graph");
        if (p.merge) { ok(f3ps_merge(ctx, p.threshold), "f3ps_merge"); tick("merge"); }
        ok(f3ps_sync(ctx), "f3ps_sync");
        cu(cudaStreamSynchronize(st), "sync");
        for (size_t i = 1; i < ev.size(); ++i) { float ms = 0; cudaEventElapsedTime(&ms, ev[i - 1].second, ev[i].second); info.stage_ms.emplace_back(ev[i].first, ms); }
        float total = 0; cudaEventElapsedTime(&total, ev.front().second, ev.back().second); info.stage_ms.emplace_back("total", total);
        info.bytes_exchanged = moved;
    } catch (const Fail& f) {
        info.error = f.what(); status_[(size_t)rank] = f.code ? f.code : F3PS_ERR_CUDA;
        // a rank that fails leaves its peers waiting in a collective: abort the communicators (once) so that every thread returns
        static std::mutex abort_mutex;
        std::lock_guard<std::mutex> l(abort_mutex);
        for (size_t r = 0; r < comm_.size(); ++r) if (comm_[r]) { ncclCommAbort((ncclComm_t)comm_[r]); comm_[r] = nullptr; }
        init_error_ = "a previous run failed: " + info.error;          // the communicators are gone; build a new SlabRun
    }
    for (auto& e : ev) cudaEventDestroy(e.second);
}

}  // namespace f3ps_host
