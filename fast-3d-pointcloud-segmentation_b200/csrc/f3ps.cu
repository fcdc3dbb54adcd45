// f3ps.cu -- host orchestration and the C ABI (include/f3ps.h) of the B200-native
// supervoxel-plus-merging path.  One handle = one device + one stream; every stage is a short
// chain of kernels on that stream; the host only waits where an array size must be known.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <map>
#include <mutex>
#include <new>
#include <set>
#include <utility>

#include "context.cuh"

using namespace f3ps;

extern "C" const unsigned char f3ps_lab_lut_begin[];   // lab_lut.S (.incbin of data/lab_lut_s16.bin)
extern "C" const unsigned char f3ps_lab_lut_end[];

namespace {

int ctx_fail(f3ps_ctx* ctx, int code, const std::string& msg) { ctx->err = msg; return code; }
int ctx_fail_cuda(f3ps_ctx* ctx, cudaError_t e, const char* what, const char* file, int line) {
    char buf[512];
    snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
    ctx->err = buf;
    return F3PS_ERR_CUDA;
}

inline int grid_for(int64_t n, int threads, int max_blocks = kSMs * 16) {
    int64_t b = (n + threads - 1) / threads;
    return (int)std::max<int64_t>(1, std::min<int64_t>(b, max_blocks));
}
inline unsigned next_pow2(unsigned v) { unsigned p = 1; while (p < v) p <<= 1; return p; }
inline int bits_for(unsigned maxval) { int b = 1; while ((maxval >> b) != 0 && b < 32) ++b; return b; }

#define LAUNCH(ctx, kernel, grid, block, smem, ...)                                         \
    do {                                                                                    \
        kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);                    \
        (ctx)->launches++;                                                                  \
        F3PS_CUDA_OK(cudaPeekAtLastError());                                                \
    } while (0)

// Wait for the handle's stream.  Spinning (cudaStreamSynchronize) has the lowest latency for one frame; a sweep with more
// frames in flight than host cores must sleep instead (blocking event), or the spinning waiters starve the launching threads.
cudaError_t wait_stream(f3ps_ctx* ctx) {
    if (!ctx->blocking_wait) return cudaStreamSynchronize(ctx->stream);
    cudaError_t e = cudaEventRecord(ctx->ev_wait, ctx->stream);
    if (e != cudaSuccess) return e;
    return cudaEventSynchronize(ctx->ev_wait);
}

int pull_scalars(f3ps_ctx* ctx) {
    F3PS_CUDA_OK(cudaMemcpyAsync(ctx->h_sc, ctx->d_sc, sizeof(DevScalars), cudaMemcpyDeviceToHost, ctx->stream));
    F3PS_CUDA_OK(wait_stream(ctx));
    return F3PS_OK;
}
#define SC(field) (&ctx->d_sc->field)

int mark(f3ps_ctx* ctx, int i) {
    F3PS_CUDA_OK(cudaEventRecord(ctx->ev[i], ctx->stream));
    ctx->ev_valid[i] = true;
    return F3PS_OK;
}

// ---- radix sort driver ------------------------------------------------------------------------
// pass 0 reads (src_k, src_v) -- src_v == nullptr means the payload is the element index -- and the
// passes ping-pong between scratch pairs A and B (A may alias the source when it can be clobbered).
template <typename KeyT>
int sort_pairs(f3ps_ctx* ctx, const KeyT* src_k, const unsigned* src_v, KeyT* a_k, unsigned* a_v, KeyT* b_k, unsigned* b_v,
               const unsigned* n_ptr, int64_t n_cap, int bits, KeyT** keys_out, unsigned** vals_out) {
    const int passes = std::max(1, (bits + kRadixBits - 1) / kRadixBits);
    const bool small = n_cap < (1 << 20);
    const int tile = kSortThreads * (small ? 4 : 16);
    const int64_t tiles = std::max<int64_t>(1, (n_cap + tile - 1) / tile);
    const size_t hist_words = (size_t)passes * kRadix;
    const size_t state_words = (size_t)passes * tiles * kRadix;
    const size_t words = hist_words + state_words + passes;
    F3PS_CUDA_OK(ctx->sort_scratch.ensure(words * 4));
    unsigned* ghist = ctx->sort_scratch.as<unsigned>();
    unsigned* state = ghist + hist_words;
    unsigned* tickets = state + state_words;
    F3PS_CUDA_OK(cudaMemsetAsync(ghist, 0, words * 4, ctx->stream));
    LAUNCH(ctx, radix_histogram_kernel<KeyT>, grid_for(n_cap, 256 * 8, kSMs * 4), 256, hist_words * 4, src_k, n_ptr, n_cap, passes, ghist);
    LAUNCH(ctx, radix_scan_hist_kernel, passes, kRadix, 0, ghist);
    const KeyT* ki = src_k; const unsigned* vi = src_v;
    KeyT* ko = a_k; unsigned* vo = a_v;
    for (int p = 0; p < passes; ++p) {
        if (small)
            LAUNCH(ctx, (radix_onesweep_kernel<KeyT, 4>), (int)tiles, kSortThreads, 0, ki, vi, ko, vo, n_ptr, n_cap, p * kRadixBits,
                   ghist + (size_t)p * kRadix, state + (size_t)p * tiles * kRadix, tickets + p);
        else
            LAUNCH(ctx, (radix_onesweep_kernel<KeyT, 16>), (int)tiles, kSortThreads, 0, ki, vi, ko, vo, n_ptr, n_cap, p * kRadixBits,
                   ghist + (size_t)p * kRadix, state + (size_t)p * tiles * kRadix, tickets + p);
        ki = ko; vi = vo;
        if (ko == a_k) { ko = b_k; vo = b_v; } else { ko = a_k; vo = a_v; }
    }
    *keys_out = const_cast<KeyT*>(ki); *vals_out = const_cast<unsigned*>(vi);
    return F3PS_OK;
}

template <typename Op>
int run_compact(f3ps_ctx* ctx, Op op, const unsigned* n_ptr, int64_t n_cap, unsigned* count) {
    const int tile = kSelThreads * kSelItems;
    const int64_t tiles = std::max<int64_t>(1, (n_cap + tile - 1) / tile);
    F3PS_CUDA_OK(ctx->compact_scratch.ensure((tiles + 1) * 4));
    unsigned* state = ctx->compact_scratch.as<unsigned>();
    F3PS_CUDA_OK(cudaMemsetAsync(state, 0, (tiles + 1) * 4, ctx->stream));
    LAUNCH(ctx, compact_kernel<Op>, (int)tiles, kSelThreads, 0, op, n_ptr, n_cap, count, state, state + tiles);
    return F3PS_OK;
}

__global__ void iota_kernel(unsigned* p, unsigned n) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = i;
}
__global__ void pos_run_kernel(const unsigned* __restrict__ sorted_label, const unsigned* __restrict__ rank_of_label, unsigned n, unsigned* __restrict__ pos_run) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned l = sorted_label[i];
        pos_run[i] = l ? rank_of_label[l] : 0xffffffffu;
    }
}
__global__ void pos_gather_kernel(const unsigned* __restrict__ order, const float4* __restrict__ vox_xyz, unsigned n, float4* __restrict__ pos_data) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) pos_data[i] = vox_xyz[order[i]];
}
__global__ void decode_edge_keys_kernel(const unsigned long long* __restrict__ compact, unsigned n, int kb, unsigned long long* __restrict__ wide) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned long long k = compact[i];
        wide[i] = ((k >> kb) << 32) | (k & ((1ull << kb) - 1ull));
    }
}
struct EdgeSlotCompactOp {      // hash-set slots -> compact keys (rank_a << kb | rank_b), unsorted
    const unsigned long long* slots; unsigned long long* keys; unsigned* vals; int kb;
    typedef int Payload;
    __device__ __forceinline__ bool test(int64_t i, Payload&) const { return slots[i] != 0ull; }
    __device__ __forceinline__ void emit(unsigned pos, int64_t i, const Payload&) const {
        const unsigned long long k = slots[i] - 1ull;
        keys[pos] = ((k >> 32) << kb) | (k & 0xffffffffull); vals[pos] = pos;
    }
};
__global__ void lab_test_kernel(const short* lut, const float* rgb, float* lab, int64_t n) {
    for (int64_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float o[3]; rgb2lab(lut, rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2], o);
        lab[3 * i] = o[0]; lab[3 * i + 1] = o[1]; lab[3 * i + 2] = o[2];
    }
}
__global__ void ciede_test_kernel(const float* l1, const float* l2, float* out, int64_t n) {
    for (int64_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = lab_ciede00(l1 + 3 * i, l2 + 3 * i);
}
__global__ void rgb_eucl_test_kernel(const float* c1, const float* c2, float* out, int64_t n) {
    for (int64_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = rgb_eucl(c1 + 3 * i, c2 + 3 * i);
}
RegionArrays carve_regions(void* base, size_t S) {
    RegionArrays R; char* p = (char*)base;
    auto take = [&](size_t bytes) { char* q = p; p += (bytes + 255) & ~(size_t)255; return q; };
    R.mean = (float4*)take(S * 16); R.accu0 = (float4*)take(S * 16); R.accu1 = (float4*)take(S * 16); R.accu2 = (float4*)take(S * 16);
    R.centroid = (float4*)take(S * 16); R.normal = (float4*)take(S * 16); R.cvec = (float4*)take(S * 16);
    R.n = (int*)take(S * 4); R.head = (int*)take(S * 4); R.tail = (int*)take(S * 4); R.next_run = (int*)take(S * 4);
    return R;
}
size_t region_bytes(size_t S) { return 7 * ((S * 16 + 255) & ~(size_t)255) + 4 * ((S * 4 + 255) & ~(size_t)255); }
EdgeArrays carve_edges(void* base, size_t E) {
    EdgeArrays A; char* p = (char*)base;
    auto take = [&](size_t bytes) { char* q = p; p += (bytes + 255) & ~(size_t)255; return q; };
    A.stamp = (long long*)take(E * 8);
    A.a = (unsigned*)take(E * 4); A.b = (unsigned*)take(E * 4); A.dc = (float*)take(E * 4); A.dg = (float*)take(E * 4); A.w = (float*)take(E * 4);
    return A;
}
size_t edge_bytes(size_t E) { return ((E * 8 + 255) & ~(size_t)255) + 5 * ((E * 4 + 255) & ~(size_t)255); }

EdgeParams edge_params(const f3ps_ctx* ctx) {
    EdgeParams ep;
    ep.color_mode = ctx->mp.color_mode; ep.geom_mode = ctx->mp.geom_mode; ep.merge_mode = ctx->mp.merge_mode;
    ep.bins = ctx->mp.bins; ep.lambda = ctx->mp.lambda;
    ep.cdf_c = ctx->cdf_c.as<float>(); ep.cdf_g = ctx->cdf_g.as<float>(); ep.lab_lut = ctx->d_lab_lut;
    return ep;
}

int need(f3ps_ctx* ctx, int level, const char* what) {
    if (ctx->progress < level) return ctx_fail(ctx, F3PS_ERR_LOGIC, std::string(what) + ": earlier stage has not run");
    return F3PS_OK;
}

// ---- K1 -------------------------------------------------------------------------------------------
template <typename KeyT>
int voxelize_typed(f3ps_ctx* ctx, PointLoader pl) {
    const int64_t N = ctx->n_points;
    F3PS_CUDA_OK(ctx->keys_a.ensure(N * sizeof(KeyT))); F3PS_CUDA_OK(ctx->keys_b.ensure(N * sizeof(KeyT)));
    F3PS_CUDA_OK(ctx->vals_a.ensure(N * 4)); F3PS_CUDA_OK(ctx->vals_b.ensure(N * 4));
    F3PS_CUDA_OK(ctx->starts.ensure((N + 1) * 4));
    KeygenOp<KeyT> kop{pl, ctx->vp.use_transform, SC(fp), ctx->keys_a.as<KeyT>(), ctx->vals_a.as<unsigned>()};
    int rc = run_compact(ctx, kop, nullptr, N, SC(n_valid));
    if (rc) return rc;
    KeyT* sk; unsigned* sv;
    rc = sort_pairs<KeyT>(ctx, ctx->keys_a.as<KeyT>(), ctx->vals_a.as<unsigned>(), ctx->keys_b.as<KeyT>(), ctx->vals_b.as<unsigned>(),
                          ctx->keys_a.as<KeyT>(), ctx->vals_a.as<unsigned>(), SC(n_valid), N, 3 * ctx->depth, &sk, &sv);
    if (rc) return rc;
    ctx->sorted_keys = sk; ctx->sorted_idx = sv;
    HeadOp<KeyT> hop{sk, ctx->starts.as<unsigned>()};
    rc = run_compact(ctx, hop, SC(n_valid), N, SC(n_voxels));
    if (rc) return rc;
    rc = pull_scalars(ctx);                                   // host needs V to size the voxel arrays
    if (rc) return rc;
    ctx->V = ctx->h_sc->n_voxels; ctx->n_valid = ctx->h_sc->n_valid;
    const size_t V = std::max(1u, ctx->V);
    F3PS_CUDA_OK(ctx->vox_xyz.ensure(V * 16)); F3PS_CUDA_OK(ctx->vox_rgb.ensure(V * 16)); F3PS_CUDA_OK(ctx->vox_key.ensure(V * 8));
    if (ctx->V)
        LAUNCH(ctx, voxel_accumulate_kernel<KeyT>, grid_for(ctx->V, 128), 128, 0, pl, sk, sv, ctx->starts.as<unsigned>(), SC(n_voxels), SC(n_valid),
               ctx->vox_xyz.as<float4>(), ctx->vox_rgb.as<float4>(), ctx->vox_key.as<uint64_t>(), ctx->point_voxel.as<int>());
    return F3PS_OK;
}

} // namespace

// =====================================================================================================
extern "C" {

const char* f3ps_version(void) { return "f3ps-b200 0.1 (sm_100a)"; }

int f3ps_create(int device, void* stream, f3ps_ctx** out) {
    if (!out) return F3PS_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    // Frames of a sweep run on independent handles / streams; the default of 8 hardware work queues would serialise
    // their persistent merge kernels 4-8 at a time.  Only effective when set before the CUDA context exists.
    setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return F3PS_ERR_CUDA;   // no CPU fallback
    f3ps_ctx* ctx = new (std::nothrow) f3ps_ctx();
    if (!ctx) return F3PS_ERR_CUDA;
    ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return F3PS_ERR_CUDA; }
    if (stream) ctx->stream = (cudaStream_t)stream;
    else { if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return F3PS_ERR_CUDA; } ctx->private_stream = ctx->stream; }
    bool ok = cudaMalloc(&ctx->d_sc, sizeof(DevScalars)) == cudaSuccess &&
              cudaMallocHost(&ctx->h_sc, sizeof(DevScalars)) == cudaSuccess;
    const size_t lut_bytes = (size_t)(f3ps_lab_lut_end - f3ps_lab_lut_begin);
    ok = ok && lut_bytes == 33 * 33 * 33 * 3 * 2 && cudaMalloc(&ctx->d_lab_lut, lut_bytes) == cudaSuccess &&
         cudaMemcpy(ctx->d_lab_lut, f3ps_lab_lut_begin, lut_bytes, cudaMemcpyHostToDevice) == cudaSuccess;
    for (int i = 0; i < f3ps_ctx::kEvents && ok; ++i) ok = cudaEventCreate(&ctx->ev[i]) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->ev_wait, cudaEventBlockingSync | cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->ev_batch, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) { f3ps_destroy(ctx); return F3PS_ERR_CUDA; }
    // the handle's stream is non-blocking: it does not wait for the legacy stream the two copies above ran on
    cudaMemsetAsync(ctx->d_sc, 0, sizeof(DevScalars), ctx->stream);
    if (cudaDeviceSynchronize() != cudaSuccess) { f3ps_destroy(ctx); return F3PS_ERR_CUDA; }
    memset(ctx->h_sc, 0, sizeof(DevScalars));
    *out = ctx;
    return F3PS_OK;
}

void f3ps_destroy(f3ps_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    // (device buffers are DevBuf members: `delete ctx` below releases every one of them)
    if (ctx->d_sc) cudaFree(ctx->d_sc);
    if (ctx->h_sc) cudaFreeHost(ctx->h_sc);
    if (ctx->d_lab_lut) cudaFree(ctx->d_lab_lut);
    for (int i = 0; i < f3ps_ctx::kEvents; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->ev_wait) cudaEventDestroy(ctx->ev_wait);
    if (ctx->ev_batch) cudaEventDestroy(ctx->ev_batch);
    if (ctx->h_batch_sc) cudaFreeHost(ctx->h_batch_sc);
    if (ctx->private_stream) cudaStreamDestroy(ctx->private_stream);
    delete ctx;
}

const char* f3ps_last_error(const f3ps_ctx* ctx) { return ctx ? ctx->err.c_str() : "null handle"; }
int64_t f3ps_launch_count(const f3ps_ctx* ctx) { return ctx ? ctx->launches : 0; }

int f3ps_set_vccs_params(f3ps_ctx* ctx, float rv, float rs, float wc, float ws, float wn, int use_transform, int fold_negative_z) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    if (!(rv > 0) || !(rs > 0)) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "resolutions must be positive");
    ctx->vp = VccsParams{rv, rs, wc, ws, wn, use_transform ? 1 : 0, fold_negative_z ? 1 : 0};
    ctx->slab_frame = false; ctx->slab_range = false;
    ctx->progress = std::min(ctx->progress, (int)P_INPUT);
    return F3PS_OK;
}

// Clustering::set_merging / set_lambda / set_bins_num, src/clustering.cpp:562-597
int f3ps_set_merge_params(f3ps_ctx* ctx, int color, int geom, int merging, float lambda, int bins) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    if (color < 0 || color > 1 || geom < 0 || geom > 1 || merging < 0 || merging > 2)
        return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "unknown distance / merging enum value");
    if (merging == F3PS_MANUAL_LAMBDA && (lambda < 0 || lambda > 1 || lambda != lambda))
        return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "Argument outside range [0, 1]");
    if (merging == F3PS_EQUALIZATION && (bins <= 0 || bins > 32767))
        return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "Argument lower than 0");
    ctx->mp = MergeParams{color, geom, merging, merging == F3PS_MANUAL_LAMBDA ? lambda : 0.5f, merging == F3PS_EQUALIZATION ? bins : 500};
    if (ctx->progress >= P_GRAPH) ctx->progress = ctx->graph_from_host ? (int)P_GRAPH - 1 : (int)P_EXPANDED;   // weights are stale
    return F3PS_OK;
}

int f3ps_set_input(f3ps_ctx* ctx, const void* points, int64_t n, int stride, int on_device) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    if (n < 0 || (stride != 16 && stride != 32) || (n > 0 && !points)) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "bad input description");
    if (n >= (1ll << 31)) return ctx_fail(ctx, F3PS_ERR_CAPACITY, "more than 2^31 points per handle");
    cudaSetDevice(ctx->device);
    if (on_device) ctx->d_points = (const uint8_t*)points;
    else {
        F3PS_CUDA_OK(ctx->in_buf.ensure(std::max<int64_t>(n, 1) * stride));
        if (n) F3PS_CUDA_OK(cudaMemcpyAsync(ctx->in_buf.p, points, (size_t)n * stride, cudaMemcpyHostToDevice, ctx->stream));
        ctx->d_points = ctx->in_buf.as<uint8_t>();
    }
    ctx->n_points = n; ctx->stride = stride;
    ctx->progress = P_INPUT; ctx->graph_from_host = false;
    return F3PS_OK;
}

int f3ps_sync(f3ps_ctx* ctx) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    F3PS_CUDA_OK(wait_stream(ctx));
    return F3PS_OK;
}

// ---- K1 -------------------------------------------------------------------------------------------
int f3ps_voxelize(f3ps_ctx* ctx) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_INPUT, "f3ps_voxelize"); if (rc) return rc;
    cudaSetDevice(ctx->device);
    rc = mark(ctx, 0); if (rc) return rc;
    const int64_t N = ctx->n_points;
    PointLoader pl{ctx->d_points, ctx->stride, ctx->vp.fold_negative_z};
    DevScalars init; memset(&init, 0, sizeof init);
    for (int a = 0; a < 3; ++a) { init.fp.ord_min[a] = 0xffffffffu; init.fp.ord_max[a] = 0u; }
    if (ctx->slab_frame) init.fp = ctx->slab_fp;
    *ctx->h_sc = init;
    F3PS_CUDA_OK(cudaMemcpyAsync(ctx->d_sc, ctx->h_sc, sizeof(DevScalars), cudaMemcpyHostToDevice, ctx->stream));
    F3PS_CUDA_OK(ctx->point_voxel.ensure(std::max<int64_t>(N, 1) * 4));
    F3PS_CUDA_OK(cudaMemsetAsync(ctx->point_voxel.p, 0xff, std::max<int64_t>(N, 1) * 4, ctx->stream));
    ctx->V = 0; ctx->n_valid = 0; ctx->depth = 0;
    ctx->slab_range = false;
    if (ctx->slab_frame) {                                    // slab mode: the frame of the WHOLE cloud, agreed on by all ranks
        ctx->depth = ctx->slab_fp.depth;
        if (N > 0 && ctx->slab_fp.any_finite) {
            rc = ctx->key64 ? voxelize_typed<uint64_t>(ctx, pl) : voxelize_typed<uint32_t>(ctx, pl);
            if (rc) return rc;
        }
    } else if (N > 0) {
        LAUNCH(ctx, bbox_kernel, grid_for(N, 256 * 4, kSMs * 8), 256, 0, pl, N, ctx->vp.use_transform, SC(fp));
        LAUNCH(ctx, frame_setup_kernel, 1, 1, 0, SC(fp), ctx->vp.voxel_res);
        rc = pull_scalars(ctx); if (rc) return rc;            // host needs the depth to pick the key width / pass count
        ctx->depth = ctx->h_sc->fp.depth;
        if (ctx->h_sc->fp.any_finite) {
            if (ctx->depth > 21) return ctx_fail(ctx, F3PS_ERR_CAPACITY, "adjacency octree depth > 21");
            ctx->key64 = 3 * ctx->depth > 32;
            rc = ctx->key64 ? voxelize_typed<uint64_t>(ctx, pl) : voxelize_typed<uint32_t>(ctx, pl);
            if (rc) return rc;
        }
    }
    ctx->progress = P_VOXELS;
    return mark(ctx, 1);
}

// ---- K2 -------------------------------------------------------------------------------------------
int f3ps_neighbors(f3ps_ctx* ctx) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_VOXELS, "f3ps_neighbors"); if (rc) return rc;
    cudaSetDevice(ctx->device);
    const unsigned V = ctx->V; const size_t Vc = std::max(1u, V);
    const unsigned cap = next_pow2(std::max(64u, 2 * V));
    ctx->hash_mask = cap - 1;
    F3PS_CUDA_OK(ctx->hash_slots.ensure((size_t)cap * 8)); F3PS_CUDA_OK(ctx->hash_vals.ensure((size_t)cap * 4));
    F3PS_CUDA_OK(ctx->nbr_row.ensure(Vc * kNbrStride * 4)); F3PS_CUDA_OK(ctx->nbr_col.ensure(Vc * 27 * 4));
    F3PS_CUDA_OK(cudaMemsetAsync(ctx->hash_slots.p, 0, (size_t)cap * 8, ctx->stream));
    if (V) {
        LAUNCH(ctx, hash_build_kernel, grid_for(V, 256), 256, 0, ctx->vox_key.as<uint64_t>(), SC(n_voxels),
               ctx->hash_slots.as<unsigned long long>(), ctx->hash_vals.as<unsigned>(), ctx->hash_mask);
        LAUNCH(ctx, neighbors_kernel, grid_for(V, 128), 128, 0, ctx->vox_key.as<uint64_t>(), SC(n_voxels), SC(fp),
               ctx->hash_slots.as<unsigned long long>(), ctx->hash_vals.as<unsigned>(), ctx->hash_mask, ctx->nbr_row.as<int>(),
               ctx->nbr_col.as<int>(), V);
    }
    ctx->progress = P_NEIGHBORS;
    return mark(ctx, 2);
}

// ---- K3 -------------------------------------------------------------------------------------------
int f3ps_normals(f3ps_ctx* ctx) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_NEIGHBORS, "f3ps_normals"); if (rc) return rc;
    cudaSetDevice(ctx->device);
    const unsigned V = ctx->V; const size_t Vc = std::max(1u, V);
    F3PS_CUDA_OK(ctx->vox_normal.ensure(Vc * 16)); F3PS_CUDA_OK(ctx->vox_curv.ensure(Vc * 4));
    const unsigned vb = ctx->slab_range ? ctx->own_begin : 0u, ve = ctx->slab_range ? ctx->own_end : 0xffffffffu;
    if (V && ve > vb)
        LAUNCH(ctx, voxel_normals_kernel, grid_for(std::min(V, ve) - vb, 128), 128, 0, ctx->vox_xyz.as<float4>(), ctx->nbr_row.as<int>(), SC(n_voxels),
               ctx->vox_normal.as<float4>(), ctx->vox_curv.as<float>(), vb, ve);
    ctx->progress = P_NORMALS;
    return mark(ctx, 3);
}

// ---- K4 -------------------------------------------------------------------------------------------
int f3ps_seeds(f3ps_ctx* ctx) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_NORMALS, "f3ps_seeds"); if (rc) return rc;
    cudaSetDevice(ctx->device);
    const unsigned V = ctx->V; const size_t Vc = std::max(1u, V);
    ctx->n_cells = 0; ctx->S0 = 0;
    DevBuf* b8[] = {&ctx->cell_code, &ctx->cell_code_b, &ctx->vox_cell, &ctx->cell_codes};
    for (DevBuf* b : b8) F3PS_CUDA_OK(b->ensure(Vc * 8));
    DevBuf* b4[] = {&ctx->cell_vox, &ctx->cell_vox_b, &ctx->cell_start, &ctx->cell_nn, &ctx->cell_keep, &ctx->seeds};
    for (DevBuf* b : b4) F3PS_CUDA_OK(b->ensure((Vc + 1) * 4));
    if (V) {
        LAUNCH(ctx, seed_box_kernel, 1, 1024, 0, ctx->vox_xyz.as<float4>(), SC(n_voxels), ctx->vp.seed_res, SC(sb));
        LAUNCH(ctx, seed_cell_kernel, grid_for(V, 256), 256, 0, ctx->vox_xyz.as<float4>(), SC(n_voxels), SC(sb), ctx->vox_cell.as<uint64_t>());
        rc = pull_scalars(ctx); if (rc) return rc;            // seed octree depth decides the sort width
        const SeedBox& sb = ctx->h_sc->sb;
        if (sb.n_events > kMaxSeedEvents) return ctx_fail(ctx, F3PS_ERR_CAPACITY, "seed octree grew more than 48 times");
        if (sb.depth > 21) return ctx_fail(ctx, F3PS_ERR_CAPACITY, "seed octree depth > 21");
        uint64_t* sc; unsigned* sv;
        rc = sort_pairs<uint64_t>(ctx, ctx->vox_cell.as<uint64_t>(), nullptr, ctx->cell_code.as<uint64_t>(), ctx->cell_vox.as<unsigned>(),
                                  ctx->cell_code_b.as<uint64_t>(), ctx->cell_vox_b.as<unsigned>(), SC(n_voxels), V, 3 * sb.depth, &sc, &sv);
        if (rc) return rc;
        HeadOp<uint64_t> hop{sc, ctx->cell_start.as<unsigned>()};
        rc = run_compact(ctx, hop, SC(n_voxels), V, SC(n_cells)); if (rc) return rc;
        LAUNCH(ctx, gather_cell_codes_kernel, grid_for(V, 256), 256, 0, sc, ctx->cell_start.as<unsigned>(), SC(n_cells), ctx->cell_codes.as<uint64_t>());
        LAUNCH(ctx, seed_select_kernel, grid_for((int64_t)V * 4, 256), 256, 0, ctx->vox_xyz.as<float4>(), ctx->vox_cell.as<uint64_t>(), sv,
               ctx->cell_start.as<unsigned>(), ctx->cell_codes.as<uint64_t>(), SC(n_cells), SC(n_voxels), SC(sb), ctx->vp.seed_res,
               ctx->vp.voxel_res, ctx->cell_nn.as<int>(), ctx->cell_keep.as<unsigned>());
        KeepOp kop{ctx->cell_keep.as<unsigned>(), ctx->cell_nn.as<int>(), ctx->seeds.as<int>()};
        rc = run_compact(ctx, kop, SC(n_cells), V, SC(n_seeds)); if (rc) return rc;
        rc = pull_scalars(ctx); if (rc) return rc;            // S0 sizes the per-label tables
        ctx->n_cells = ctx->h_sc->n_cells; ctx->S0 = ctx->h_sc->n_seeds;
    }
    ctx->progress = P_SEEDS;
    return mark(ctx, 4);
}

// ---- K5 -------------------------------------------------------------------------------------------
// One cooperative launch runs createSupervoxelHelpers, every expansion round and makeSupervoxels' lists
// (kernels_expand.cuh); the host only learns the number of surviving helpers afterwards.
// Sweeps: cooperative launches run ONE AT A TIME on a device (measured: K5 of concurrent frames serialises at its solo
// duration, 0.74 ms per frame, while K1..K4 and K6 scale with the streams), so a sweep may cap the cooperative grid
// (f3ps_set_expand_sharing) or run K5 as one thread-block cluster per frame (f3ps_set_expand_kernel).

static int expand_prepare(f3ps_ctx* ctx, ExpandArgs& A) {
    const unsigned V = ctx->V, S0 = ctx->S0; const size_t Vc = std::max(1u, V), Sc = (size_t)S0 + 2, Lc = Vc + Sc;
    DevBuf* bv[] = {&ctx->own_a, &ctx->own_b, &ctx->dst_a, &ctx->dst_b, &ctx->st0, &ctx->st1, &ctx->owner0, &ctx->dist0};
    for (DevBuf* b : bv) F3PS_CUDA_OK(b->ensure(Vc * 4));
    F3PS_CUDA_OK(ctx->phantom.ensure(Vc * 4 * kPhSlots));
    DevBuf* bl[] = {&ctx->lab_keys_a, &ctx->lab_vals_a, &ctx->lab_vals_b};
    for (DevBuf* b : bl) F3PS_CUDA_OK(b->ensure(Lc * 4));
    F3PS_CUDA_OK(ctx->chg_a.ensure(Vc)); F3PS_CUDA_OK(ctx->chg_b.ensure(Vc));
    DevBuf* bs[] = {&ctx->seg_start, &ctx->seg_end, &ctx->lab_count, &ctx->lab_count2, &ctx->lab_fill, &ctx->phantom_leaf, &ctx->sv_label, &ctx->rank_of_label};
    for (DevBuf* b : bs) F3PS_CUDA_OK(b->ensure(Sc * 4));
    F3PS_CUDA_OK(ctx->cen_xyz.ensure(Sc * 16)); F3PS_CUDA_OK(ctx->cen_rgb.ensure(Sc * 16)); F3PS_CUDA_OK(ctx->cen_nrm.ensure(Sc * 16));
    const int max_depth = (int)(1.8f * ctx->vp.seed_res / ctx->vp.voxel_res);     // SupervoxelClustering::extract
    ctx->rounds = std::max(0, max_depth - 1);
    F3PS_CUDA_OK(cudaMemsetAsync(SC(xctl), 0, sizeof(ExpandCtl), ctx->stream));
    ctx->sorted_label = ctx->lab_keys_a.as<unsigned>(); ctx->sorted_vox = ctx->lab_vals_b.as<unsigned>();
    A.nbr_col = ctx->nbr_col.as<int>(); A.nbr_row = ctx->nbr_row.as<int>(); A.V_cap = V;
    A.vox_xyz = ctx->vox_xyz.as<float4>(); A.vox_rgb = ctx->vox_rgb.as<float4>(); A.vox_nrm = ctx->vox_normal.as<float4>();
    A.seeds = ctx->seeds.as<int>(); A.V = V; A.S0 = S0; A.rounds = ctx->rounds; A.P = ctx->vp; A.keep_centroids = 0;
    A.owner[0] = ctx->own_a.as<unsigned>(); A.owner[1] = ctx->own_b.as<unsigned>();
    A.dist[0] = ctx->dst_a.as<float>(); A.dist[1] = ctx->dst_b.as<float>();
    A.st[0] = ctx->st0.as<unsigned>(); A.st[1] = ctx->st1.as<unsigned>();
    A.chg[0] = ctx->chg_a.as<unsigned char>(); A.chg[1] = ctx->chg_b.as<unsigned char>();
    A.phantom = ctx->phantom.as<unsigned>(); A.phantom_leaf = ctx->phantom_leaf.as<int>();
    A.cen = Centroids{ctx->cen_xyz.as<float4>(), ctx->cen_rgb.as<float4>(), ctx->cen_nrm.as<float4>()};
    A.count[0] = ctx->lab_count.as<unsigned>(); A.count[1] = ctx->lab_count2.as<unsigned>(); A.fill = ctx->lab_fill.as<unsigned>(); A.off = ctx->seg_start.as<unsigned>();
    A.list_raw = ctx->lab_vals_a.as<unsigned>(); A.list_sorted = ctx->lab_vals_b.as<unsigned>(); A.pos_label = ctx->lab_keys_a.as<unsigned>();
    A.labels_out = ctx->owner0.as<unsigned>(); A.dist_out = ctx->dist0.as<float>();
    A.seg_end = ctx->seg_end.as<unsigned>(); A.sv_label = ctx->sv_label.as<unsigned>(); A.rank_of_label = ctx->rank_of_label.as<unsigned>();
    A.ctl = SC(xctl);
    return F3PS_OK;
}

static int expand_finish(f3ps_ctx* ctx) {
    int rc = pull_scalars(ctx); if (rc) return rc;
    const ExpandCtl& x = ctx->h_sc->xctl;
    if (x.error & EXPAND_ERR_TRIPLE) return ctx_fail(ctx, F3PS_ERR_CAPACITY, "more than four seed cells elected the same voxel (not modelled)");
    if (x.error & EXPAND_ERR_CAND) return ctx_fail(ctx, F3PS_ERR_CAPACITY, "more than 32 candidate helpers around one voxel");
    if (x.error & EXPAND_ERR_SWEEPS) return ctx_fail(ctx, F3PS_ERR_NOT_CONVERGED, "expansion fixed point not reached within 32 sweeps");
    ctx->S = ctx->V ? x.n_sv : 0; ctx->n_pos = ctx->V ? x.n_pos : 0;
    ctx->progress = P_EXPANDED;
    return mark(ctx, 5);
}

static int expand_launch(f3ps_ctx* ctx, bool keep_centroids) {
    const unsigned V = ctx->V;
    ExpandArgs A;
    int rc = expand_prepare(ctx, A); if (rc) return rc;
    A.keep_centroids = keep_centroids ? 1 : 0;
    if (keep_centroids) A.seeds = ctx->seeds_refine.as<int>();      // the seed voxels of f3ps_seeds stay what f3ps_get_seeds returns
    const bool cluster = V && ctx->expand_kernel_choice == 2;      // sweeps ask for it (f3ps_set_expand_kernel); one frame alone is fastest on the cooperative grid
    if (cluster) {
        // one thread-block cluster per frame (kernels_expand.cuh): ~2 voxels per thread, at most 16 CTAs
        int ncta = (int)std::min<int64_t>(kExpandClusterMax, ((int64_t)V + 2 * kExpandClusterThreads - 1) / (2 * kExpandClusterThreads));
        if (ctx->expand_cluster_ctas > 0) ncta = std::min(ncta, ctx->expand_cluster_ctas);
        ncta = std::max(1, ncta);
        if (!ctx->expand_cluster_attr_set) {
            F3PS_CUDA_OK(cudaFuncSetAttribute((const void*)expand_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
            ctx->expand_cluster_attr_set = true;
        }
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(ncta); cfg.blockDim = dim3(kExpandClusterThreads); cfg.dynamicSmemBytes = 0; cfg.stream = ctx->stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension; attr[0].val.clusterDim.x = (unsigned)ncta; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        F3PS_CUDA_OK(cudaLaunchKernelEx(&cfg, expand_cluster_kernel, A));
        ctx->launches++;
        return expand_finish(ctx);
    }
    if (V) {
        if (!ctx->expand_blocks_per_sm) {
            int nb = 0;
            F3PS_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, expand_persistent_kernel, kExpandThreads, 0));
            int sms = 0;
            F3PS_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
            ctx->expand_blocks_per_sm = std::max(1, nb); ctx->sm_count = std::max(1, sms);
        }
        const int64_t want = ((int64_t)V + kExpandThreads - 1) / kExpandThreads;
        int grid = (int)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)std::min(ctx->expand_blocks_per_sm, 2) * ctx->sm_count));
        if (ctx->expand_ctas > 0) grid = std::min(grid, ctx->expand_ctas);   // sweeps: fewer CTAs per frame, more frames side by side
        void* args[] = {&A};
        F3PS_CUDA_OK(cudaLaunchCooperativeKernel((const void*)expand_persistent_kernel, dim3(grid), dim3(kExpandThreads), args, 0, ctx->stream));
        ctx->launches++;
    }
    return expand_finish(ctx);
}

int f3ps_expand(f3ps_ctx* ctx) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_SEEDS, "f3ps_expand"); if (rc) return rc;
    cudaSetDevice(ctx->device);
    return expand_launch(ctx, false);
}

// pcl::SupervoxelClustering::refineSupervoxels(num_itr, ...): per iteration refineNormals, reseedSupervoxels and the expansion
// rounds again, starting from the helpers' current centroids (kernels_vccs.cuh, kernels_expand.cuh).  Leaves the handle where
// f3ps_expand leaves it: labels, distances, voxel normals and the supervoxels are the refined ones, the graph has to be rebuilt.
int f3ps_refine(f3ps_ctx* ctx, int num_itr) {
    if (!ctx || num_itr < 0) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_EXPANDED, "f3ps_refine"); if (rc) return rc;          // PCL: "Supervoxels must be extracted before they can be refined"
    if (ctx->graph_from_host) return ctx_fail(ctx, F3PS_ERR_LOGIC, "f3ps_refine needs the voxels of f3ps_extract, not a graph set with f3ps_set_graph");
    if (ctx->slab_range) return ctx_fail(ctx, F3PS_ERR_LOGIC, "f3ps_refine is not available in slab mode");
    cudaSetDevice(ctx->device);
    const unsigned V = ctx->V, S0 = ctx->S0;
    F3PS_CUDA_OK(ctx->seeds_refine.ensure(((size_t)S0 + 1) * 4));
    for (int it = 0; it < num_itr && V && S0; ++it) {
        LAUNCH(ctx, refine_normals_kernel, grid_for(V, 128), 128, 0, ctx->vox_xyz.as<float4>(), ctx->nbr_row.as<int>(), SC(n_voxels),
               ctx->owner0.as<unsigned>(), ctx->phantom.as<unsigned>(), ctx->vox_normal.as<float4>(), ctx->vox_curv.as<float>());
        LAUNCH(ctx, reseed_kernel, (int)std::min<unsigned>(S0, 4u * kSMs), 256, 0, ctx->cen_xyz.as<float4>(), S0, ctx->vox_xyz.as<float4>(), SC(n_voxels),
               ctx->seeds_refine.as<int>());
        ctx->progress = P_SEEDS;
        rc = expand_launch(ctx, true); if (rc) return rc;
    }
    ctx->progress = P_EXPANDED;
    return F3PS_OK;
}

// ---- K6 -------------------------------------------------------------------------------------------
static int init_weights(f3ps_ctx* ctx, unsigned E_cap) {     // Clustering::init_weights on R0 / E0 + the edge keys
    EdgeParams ep = edge_params(ctx);
    const float* lambda_dev = nullptr;
    F3PS_CUDA_OK(ctx->dbits_a.ensure((size_t)E_cap * 4)); F3PS_CUDA_OK(ctx->dbits_b.ensure((size_t)E_cap * 4));
    F3PS_CUDA_OK(ctx->dbits_c.ensure((size_t)E_cap * 4)); F3PS_CUDA_OK(ctx->dbits_d.ensure((size_t)E_cap * 4));
    F3PS_CUDA_OK(ctx->edge_vals_a.ensure((size_t)E_cap * 4)); F3PS_CUDA_OK(ctx->edge_vals_b.ensure((size_t)E_cap * 4));
    F3PS_CUDA_OK(ctx->cdf_c.ensure((size_t)std::max(1, ctx->mp.bins) * 4)); F3PS_CUDA_OK(ctx->cdf_g.ensure((size_t)std::max(1, ctx->mp.bins) * 4));
    ep.cdf_c = ctx->cdf_c.as<float>(); ep.cdf_g = ctx->cdf_g.as<float>();
    LAUNCH(ctx, region_cvec_kernel, grid_for(std::max(1u, ctx->S), 256), 256, 0, SC(xctl.n_sv), ctx->R0, ep);
    LAUNCH(ctx, edge_delta_kernel, grid_for(E_cap, 128), 128, 0, ctx->sorted_edge_keys, SC(n_edges), ctx->R0, ep, ctx->E0,
           ctx->dbits_a.as<unsigned>(), ctx->dbits_c.as<unsigned>());
    if (ctx->mp.merge_mode == F3PS_ADAPTIVE_LAMBDA && E_cap <= 16384u) {
        const unsigned n_pow2 = next_pow2(std::max(2u, E_cap));
        if (!ctx->lambda_attr_set) {
            F3PS_CUDA_OK(cudaFuncSetAttribute(adaptive_lambda_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 * 4));
            ctx->lambda_attr_set = true;
        }
        LAUNCH(ctx, adaptive_lambda_smem_kernel, 2, 1024, (size_t)n_pow2 * 4, ctx->E0.dc, ctx->E0.dg, SC(n_edges), n_pow2, SC(padf[0]), SC(pad0), SC(lambda));
        lambda_dev = SC(lambda);
    } else if (ctx->mp.merge_mode == F3PS_ADAPTIVE_LAMBDA) {
        unsigned *sc, *sg, *dummy;
        int rc = sort_pairs<unsigned>(ctx, ctx->dbits_a.as<unsigned>(), nullptr, ctx->dbits_b.as<unsigned>(), ctx->edge_vals_a.as<unsigned>(),
                                      ctx->dbits_a.as<unsigned>(), ctx->edge_vals_b.as<unsigned>(), SC(n_edges), E_cap, 32, &sc, &dummy);
        if (rc) return rc;
        rc = sort_pairs<unsigned>(ctx, ctx->dbits_c.as<unsigned>(), nullptr, ctx->dbits_d.as<unsigned>(), ctx->edge_vals_a.as<unsigned>(),
                                  ctx->dbits_c.as<unsigned>(), ctx->edge_vals_b.as<unsigned>(), SC(n_edges), E_cap, 32, &sg, &dummy);
        if (rc) return rc;
        LAUNCH(ctx, adaptive_lambda_kernel, 1, 64, 0, sc, sg, SC(n_edges), SC(lambda));
        lambda_dev = SC(lambda);
    } else if (ctx->mp.merge_mode == F3PS_EQUALIZATION) {
        const int bins = ctx->mp.bins;
        F3PS_CUDA_OK(ctx->cdf_hist.ensure((size_t)2 * bins * 4));
        LAUNCH(ctx, cdf_kernel, 2, 1024, bins <= 8192 ? (size_t)bins * 4 : 0, ctx->E0.dc, ctx->E0.dg, SC(n_edges), bins, ctx->cdf_c.as<float>(),
               ctx->cdf_g.as<float>(), ctx->cdf_hist.as<unsigned>(), SC(bad_bin));
    }
    if (ctx->mp.merge_mode != F3PS_ADAPTIVE_LAMBDA) {
        const float lam = ctx->mp.lambda;
        F3PS_CUDA_OK(cudaMemcpyAsync(SC(lambda), &lam, 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    LAUNCH(ctx, edge_weight_kernel, grid_for(E_cap, 256), 256, 0, SC(n_edges), ep, lambda_dev, ctx->E0, SC(nan_weights_init));
    return F3PS_OK;
}

int f3ps_graph(f3ps_ctx* ctx) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    cudaSetDevice(ctx->device);
    if (ctx->graph_from_host) {                                // weights only (parameters changed after f3ps_set_graph)
        int rc = need(ctx, P_GRAPH - 1, "f3ps_graph"); if (rc) return rc;
        F3PS_CUDA_OK(cudaMemsetAsync(SC(nan_weights_init), 0, 4, ctx->stream));
        rc = init_weights(ctx, std::max(1u, ctx->E)); if (rc) return rc;
        ctx->progress = P_GRAPH;
        return F3PS_OK;
    }
    int rc = need(ctx, P_EXPANDED, "f3ps_graph"); if (rc) return rc;
    const unsigned V = ctx->V, S = ctx->S; const size_t Sc = std::max(1u, S), Vc = std::max(1u, V);
    F3PS_CUDA_OK(ctx->reg_init.ensure(region_bytes(Sc))); F3PS_CUDA_OK(ctx->reg_work.ensure(region_bytes(Sc)));
    ctx->R0 = carve_regions(ctx->reg_init.p, Sc); ctx->R1 = carve_regions(ctx->reg_work.p, Sc);
    F3PS_CUDA_OK(ctx->run_start.ensure(Sc * 4)); F3PS_CUDA_OK(ctx->run_end.ensure(Sc * 4)); F3PS_CUDA_OK(ctx->pos_run.ensure((Vc + Sc) * 4));
    Centroids cen{ctx->cen_xyz.as<float4>(), ctx->cen_rgb.as<float4>(), ctx->cen_nrm.as<float4>()};
    ctx->order = ctx->sorted_vox; ctx->gxyz = ctx->vox_xyz.as<float4>();
    const unsigned P = ctx->n_pos;
    const unsigned set_cap = next_pow2(std::max(1024u, 32 * S));
    ctx->edge_set_mask = set_cap - 1; ctx->edge_kb = bits_for(std::max(1u, S));
    F3PS_CUDA_OK(ctx->edge_set.ensure((size_t)set_cap * 8));
    F3PS_CUDA_OK(ctx->edge_keys_a.ensure((size_t)set_cap * 8)); F3PS_CUDA_OK(ctx->edge_keys_b.ensure((size_t)set_cap * 8));
    F3PS_CUDA_OK(ctx->edge_vals_a.ensure((size_t)set_cap * 4)); F3PS_CUDA_OK(ctx->edge_vals_b.ensure((size_t)set_cap * 4));
    F3PS_CUDA_OK(ctx->edge_init.ensure(edge_bytes(set_cap))); F3PS_CUDA_OK(ctx->edge_work.ensure(edge_bytes(set_cap)));
    ctx->E0 = carve_edges(ctx->edge_init.p, set_cap); ctx->E1 = carve_edges(ctx->edge_work.p, set_cap);
    F3PS_CUDA_OK(cudaMemsetAsync(ctx->edge_set.p, 0, (size_t)set_cap * 8, ctx->stream));
    F3PS_CUDA_OK(cudaMemsetAsync(SC(n_edges), 0, 4, ctx->stream));
    F3PS_CUDA_OK(cudaMemsetAsync(SC(edge_overflow), 0, 16, ctx->stream));   // edge_overflow, bad_bin, nan_weights_init, pad
    if (V && S) {
        LAUNCH(ctx, pos_run_kernel, grid_for(P, 256), 256, 0, ctx->sorted_label, ctx->rank_of_label.as<unsigned>(), P, ctx->pos_run.as<unsigned>());
        F3PS_CUDA_OK(ctx->pos_data_buf.ensure((size_t)std::max(1u, P) * 16));
        LAUNCH(ctx, pos_gather_kernel, grid_for(P, 256), 256, 0, ctx->sorted_vox, ctx->vox_xyz.as<float4>(), P, ctx->pos_data_buf.as<float4>());
        ctx->pos_data = ctx->pos_data_buf.as<float4>();
        LAUNCH(ctx, region_init_kernel, grid_for((int64_t)S * 32, 256), 256, 0, ctx->sv_label.as<unsigned>(), SC(xctl.n_sv), ctx->seg_start.as<unsigned>(),
               ctx->seg_end.as<unsigned>(), ctx->sorted_vox, ctx->vox_xyz.as<float4>(), cen, ctx->R0, ctx->run_start.as<unsigned>(),
               ctx->run_end.as<unsigned>());
        LAUNCH(ctx, edge_collect_kernel, grid_for(P, 256), 256, 0, ctx->nbr_col.as<int>(), V, ctx->nbr_row.as<int>(), P, ctx->sorted_label, ctx->sorted_vox,
               ctx->owner0.as<unsigned>(), ctx->rank_of_label.as<unsigned>(), ctx->edge_set.as<unsigned long long>(), ctx->edge_set_mask, SC(edge_overflow));
        EdgeSlotCompactOp sop{ctx->edge_set.as<unsigned long long>(), ctx->edge_keys_a.as<unsigned long long>(), ctx->edge_vals_a.as<unsigned>(), ctx->edge_kb};
        rc = run_compact(ctx, sop, nullptr, set_cap, SC(n_edges)); if (rc) return rc;
        unsigned long long* sk; unsigned* sv;
        rc = sort_pairs<unsigned long long>(ctx, ctx->edge_keys_a.as<unsigned long long>(), nullptr, ctx->edge_keys_b.as<unsigned long long>(),
                                            ctx->edge_vals_b.as<unsigned>(), ctx->edge_keys_a.as<unsigned long long>(), ctx->edge_vals_a.as<unsigned>(),
                                            SC(n_edges), set_cap, 2 * ctx->edge_kb, &sk, &sv);
        if (rc) return rc;
        unsigned long long* wide = (sk == ctx->edge_keys_a.as<unsigned long long>()) ? ctx->edge_keys_b.as<unsigned long long>()
                                                                                      : ctx->edge_keys_a.as<unsigned long long>();
        rc = pull_scalars(ctx); if (rc) return rc;             // E (and the overflow flag) before the weights
        if (ctx->h_sc->edge_overflow) return ctx_fail(ctx, F3PS_ERR_CAPACITY, "supervoxel edge set overflow");
        ctx->E = ctx->h_sc->n_edges;
        if (ctx->E) {
            LAUNCH(ctx, decode_edge_keys_kernel, grid_for(ctx->E, 256), 256, 0, sk, ctx->E, ctx->edge_kb, wide);
            ctx->sorted_edge_keys = wide;
            rc = init_weights(ctx, ctx->E); if (rc) return rc;
        }
    } else ctx->E = 0;
    ctx->progress = P_GRAPH;
    return mark(ctx, 6);
}

int f3ps_set_graph(f3ps_ctx* ctx, int64_t n_voxels, const float* voxel_xyz, const uint32_t* voxel_rgba, int32_t n_sv, const uint32_t* labels,
                   const int64_t* voxel_offsets, const float* centroids_xyz, const float* normals_xyz, int64_t n_adj, const uint32_t* adj_pairs) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    if (n_voxels < 0 || n_sv < 0 || n_adj < 0) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "negative size");
    cudaSetDevice(ctx->device);
    const unsigned V = (unsigned)n_voxels, S = (unsigned)n_sv;
    // supervoxels by ascending label (std::map order), voxel ranges regrouped accordingly
    std::vector<int> perm(S);
    for (unsigned s = 0; s < S; ++s) perm[s] = (int)s;
    std::sort(perm.begin(), perm.end(), [&](int x, int y) { return labels[x] < labels[y]; });
    std::map<uint32_t, unsigned> rank;
    std::vector<float4> h_xyz(std::max(1u, V));
    std::vector<unsigned> h_start(std::max(1u, S)), h_end(std::max(1u, S)), h_label(std::max(1u, S)), h_posrun(std::max(1u, V)), h_vin(std::max(1u, V));
    std::vector<float4> h_cen(std::max(1u, S)), h_nrm(std::max(1u, S));
    unsigned pos = 0;
    for (unsigned r = 0; r < S; ++r) {
        const int s = perm[r];
        if (rank.count(labels[s])) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "duplicate supervoxel label");
        rank[labels[s]] = r; h_label[r] = labels[s];
        h_start[r] = pos;
        for (int64_t i = voxel_offsets[s]; i < voxel_offsets[s + 1]; ++i, ++pos) {
            float w; uint32_t c = voxel_rgba[i] & 0x00ffffffu; memcpy(&w, &c, 4);
            h_xyz[pos] = make_float4(voxel_xyz[3 * i], voxel_xyz[3 * i + 1], voxel_xyz[3 * i + 2], w);
            h_posrun[pos] = r; h_vin[pos] = (unsigned)i;
        }
        h_end[r] = pos;
        h_cen[r] = make_float4(centroids_xyz[3 * s], centroids_xyz[3 * s + 1], centroids_xyz[3 * s + 2], 0.0f);
        h_nrm[r] = make_float4(normals_xyz[3 * s], normals_xyz[3 * s + 1], normals_xyz[3 * s + 2], 0.0f);
    }
    if (pos != V) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "voxel offsets do not cover the voxel arrays");
    // clear_adjacency keeps first <= second (src/clustering.cpp:476-486); iteration order = insertion order of the weights
    std::vector<unsigned long long> h_keys;
    for (int64_t i = 0; i < n_adj; ++i) {
        const uint32_t a = adj_pairs[2 * i], b = adj_pairs[2 * i + 1];
        if (a > b) continue;
        if (a == b) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "self-adjacent supervoxel");
        auto ia = rank.find(a), ib = rank.find(b);
        if (ia == rank.end() || ib == rank.end()) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "adjacency names an unknown label");   // map::at
        h_keys.push_back(((unsigned long long)ia->second << 32) | ib->second);
    }
    const unsigned E = (unsigned)h_keys.size();
    const size_t Sc = std::max(1u, S), Vc = std::max(1u, V), Ec = std::max(1u, E);
    F3PS_CUDA_OK(ctx->vox_xyz.ensure(Vc * 16)); F3PS_CUDA_OK(ctx->lab_vals_a.ensure(Vc * 4)); F3PS_CUDA_OK(ctx->pos_run.ensure(Vc * 4));
    F3PS_CUDA_OK(ctx->graph_vox.ensure(Vc * 4));
    F3PS_CUDA_OK(ctx->run_start.ensure(Sc * 4)); F3PS_CUDA_OK(ctx->run_end.ensure(Sc * 4)); F3PS_CUDA_OK(ctx->sv_label.ensure(Sc * 4));
    F3PS_CUDA_OK(ctx->reg_init.ensure(region_bytes(Sc))); F3PS_CUDA_OK(ctx->reg_work.ensure(region_bytes(Sc)));
    ctx->R0 = carve_regions(ctx->reg_init.p, Sc); ctx->R1 = carve_regions(ctx->reg_work.p, Sc);
    F3PS_CUDA_OK(ctx->edge_init.ensure(edge_bytes(Ec))); F3PS_CUDA_OK(ctx->edge_work.ensure(edge_bytes(Ec)));
    ctx->E0 = carve_edges(ctx->edge_init.p, Ec); ctx->E1 = carve_edges(ctx->edge_work.p, Ec);
    F3PS_CUDA_OK(ctx->edge_keys_a.ensure(Ec * 8));
    auto up = [&](void* d, const void* h, size_t bytes) { return bytes ? cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, ctx->stream) : cudaSuccess; };
    F3PS_CUDA_OK(up(ctx->vox_xyz.p, h_xyz.data(), (size_t)V * 16)); F3PS_CUDA_OK(up(ctx->pos_run.p, h_posrun.data(), (size_t)V * 4));
    F3PS_CUDA_OK(up(ctx->graph_vox.p, h_vin.data(), (size_t)V * 4));
    F3PS_CUDA_OK(up(ctx->run_start.p, h_start.data(), (size_t)S * 4)); F3PS_CUDA_OK(up(ctx->run_end.p, h_end.data(), (size_t)S * 4));
    F3PS_CUDA_OK(up(ctx->sv_label.p, h_label.data(), (size_t)S * 4));
    F3PS_CUDA_OK(up(ctx->R0.centroid, h_cen.data(), (size_t)S * 16)); F3PS_CUDA_OK(up(ctx->R0.normal, h_nrm.data(), (size_t)S * 16));
    F3PS_CUDA_OK(up(ctx->edge_keys_a.p, h_keys.data(), (size_t)E * 8));
    DevScalars init; memset(&init, 0, sizeof init);
    init.n_voxels = V; init.xctl.n_sv = S; init.n_edges = E;
    *ctx->h_sc = init;
    F3PS_CUDA_OK(cudaMemcpyAsync(ctx->d_sc, ctx->h_sc, sizeof(DevScalars), cudaMemcpyHostToDevice, ctx->stream));
    if (V) LAUNCH(ctx, iota_kernel, grid_for(V, 256), 256, 0, ctx->lab_vals_a.as<unsigned>(), V);
    if (S) LAUNCH(ctx, region_init_ranges_kernel, grid_for((int64_t)S * 32, 256), 256, 0, S, ctx->run_start.as<unsigned>(), ctx->run_end.as<unsigned>(),
                  ctx->lab_vals_a.as<unsigned>(), ctx->vox_xyz.as<float4>(), ctx->R0);
    ctx->V = V; ctx->S = S; ctx->S0 = S; ctx->E = E; ctx->n_pos = V;
    ctx->order = ctx->lab_vals_a.as<unsigned>(); ctx->sorted_vox = ctx->lab_vals_a.as<unsigned>(); ctx->gxyz = ctx->vox_xyz.as<float4>();
    ctx->pos_data = ctx->vox_xyz.as<float4>();               // identity order
    ctx->sorted_edge_keys = ctx->edge_keys_a.as<unsigned long long>();
    ctx->graph_from_host = true;
    ctx->progress = P_GRAPH - 1;
    F3PS_CUDA_OK(cudaStreamSynchronize(ctx->stream));        // host staging vectors go out of scope
    return f3ps_graph(ctx);
}

// ---- K7 -------------------------------------------------------------------------------------------
extern "C++" {
namespace {
// edge capacity of the resident kernel's tables: E rounded up to whole blocks of 32 edges (0 = more than 32 blocks per worker warp)
unsigned lean_ecap_for(unsigned E, int threads = kFastThreads) {
    const unsigned owners = (unsigned)(threads - 32 * kLeanRoleWarps);
    const unsigned nb = std::max(1u, (E + owners - 1u) / owners);
    return nb <= 32u ? std::max(32u, (E + 31u) & ~31u) : 0u;
}
// adjacency pool of the resident kernel (edge ids, 2 bytes each): the initial lists plus room for the lists that outgrow their block
constexpr size_t kLeanPoolSlack = 1u << 20;
constexpr size_t kSmemMax = 227u * 1024u;
// The opt-in to > 48 KB of dynamic shared memory is per function AND per device: remember it per (device, function).
int smem_opt_in(f3ps_ctx* ctx, const void* kern, size_t bytes) {
    static std::mutex m;
    static std::set<std::pair<int, const void*>> done;
    std::lock_guard<std::mutex> l(m);
    if (done.count({ctx->device, kern})) return F3PS_OK;
    F3PS_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    done.insert({ctx->device, kern});
    return F3PS_OK;
}
// Which kernel replays a handle's merges.  The kinds carry the merge_path of a replay that stays on one kernel.
enum MergeKind { kMergeShared = 1, kMergeGeneral = 2, kMergeL2 = 3 };
struct MergePlan {
    MergeKind kind;
    bool prof;               // resident kernel built with phase counters (kernel choice 4 / 5)
    bool to_l2;              // kMergeShared: a merge with more adjacency entries than worker threads continues on the L2 variant
    int threads; unsigned S_cap, E_cap; size_t smem;     // resident kernel: block size, table capacities, dynamic shared memory
};
// the resident kernel with its big tables in global memory, for graphs that do not fit an SM (16-bit region ids, 32-bit edge ids;
// 16 bytes of shared memory per block of 32 edges bound E near 380,000)
MergePlan plan_l2(const f3ps_ctx* ctx) {
    const unsigned S = ctx->S, E = ctx->E;
    MergePlan p{kMergeL2, ctx->merge_kernel_choice == 5, false, kFastThreads, (S + 7u) & ~7u, (E + 31u) & ~31u, 0};
    p.smem = FastSmem(nullptr, p.S_cap, p.E_cap, (char*)16).bytes;
    if (ctx->n_pos == 0 || S >= 65535u || p.E_cap > (1u << 20) || p.smem > kSmemMax) p.kind = kMergeGeneral;
    return p;
}
MergePlan plan_merge(const f3ps_ctx* ctx) {
    const unsigned S = ctx->S, E = ctx->E; const int choice = ctx->merge_kernel_choice;
    MergePlan l2 = plan_l2(ctx);
    if (choice == 2) l2.kind = kMergeGeneral;
    // the resident kernel with its tables in shared memory when the graph fits one SM (kernels_merge_lean.cuh)
    const unsigned S_cap = (S + 7u) & ~7u, E_cap = lean_ecap_for(E);
    if (choice == 2 || choice == 3 || choice == 5 || !E_cap || S > 4096u || ctx->n_pos == 0) return l2;
    const size_t smem = FastSmem(nullptr, S_cap, E_cap).bytes;
    if (smem > kSmemMax) return l2;
    // one frame alone runs the 768-thread build (80 registers) when its edges fit 21 worker warps and a merge wider than its 672
    // worker threads can continue on the L2 variant
    const bool to_l2 = l2.kind == kMergeL2, solo = to_l2 && lean_ecap_for(E, kFastThreadsSolo) != 0u;
    return MergePlan{kMergeShared, choice == 4, to_l2, solo ? kFastThreadsSolo : kFastThreads, S_cap, E_cap, smem};
}
// cluster(float) restarts from initial_state (src/clustering.cpp:678): working regions and edges, merge counters
int merge_restart(f3ps_ctx* ctx) {
    F3PS_CUDA_OK(cudaMemcpyAsync(ctx->reg_work.p, ctx->reg_init.p, region_bytes(std::max(1u, ctx->S)), cudaMemcpyDeviceToDevice, ctx->stream));
    F3PS_CUDA_OK(cudaMemcpyAsync(ctx->edge_work.p, ctx->edge_init.p, std::min(ctx->edge_init.cap, ctx->edge_work.cap), cudaMemcpyDeviceToDevice, ctx->stream));
    F3PS_CUDA_OK(cudaMemsetAsync(SC(mctl), 0, sizeof(MergeCtl), ctx->stream));
    return F3PS_OK;
}
// start of a replay: restart, merge log, output buffers
int merge_begin(f3ps_ctx* ctx) {
    int rc = mark(ctx, 7); if (rc) return rc;
    ctx->lv_thr.clear(); ctx->lv_built = 0;
    ctx->seg_points.level = ctx->seg_voxels.level = -1;
    if ((rc = merge_restart(ctx))) return rc;
    const size_t Sc = std::max(1u, ctx->S), Pc = std::max(1u, ctx->n_pos);
    F3PS_CUDA_OK(ctx->mlog.ensure(Sc * 20));
    char* lp = (char*)ctx->mlog.p;
    ctx->ML.a = (unsigned*)lp; ctx->ML.b = (unsigned*)(lp + Sc * 4); ctx->ML.w = (float*)(lp + Sc * 8);
    ctx->ML.edges_left = (unsigned*)(lp + Sc * 12); ctx->ML.regions_left = (unsigned*)(lp + Sc * 16);
    F3PS_CUDA_OK(ctx->run_out_off.ensure(Sc * 4)); F3PS_CUDA_OK(ctx->run_dense.ensure(Sc * 4)); F3PS_CUDA_OK(ctx->region_dense.ensure(Sc * 4));
    F3PS_CUDA_OK(ctx->out_xyz.ensure(Pc * 12)); F3PS_CUDA_OK(ctx->out_label.ensure(Pc * 4)); F3PS_CUDA_OK(ctx->out_voxel.ensure(Pc * 4));
    F3PS_CUDA_OK(ctx->vox_segment.ensure(Pc * 4));
    F3PS_CUDA_OK(cudaMemsetAsync(ctx->vox_segment.p, 0xff, Pc * 4, ctx->stream));
    F3PS_CUDA_OK(cudaMemsetAsync(SC(n_out), 0, 4, ctx->stream));
    return F3PS_OK;
}
// the resident kernel's arguments for one frame; resume: continue from the state in the working arrays (counters in mctl)
int fast_args(f3ps_ctx* ctx, const MergePlan& p, float threshold, bool resume, FastArgs& A) {
    const bool big = p.kind == kMergeL2;
    A.R = ctx->R1; A.E = ctx->E1; A.n_edges_ptr = SC(n_edges); A.n_sv_ptr = SC(xctl.n_sv); A.ep = edge_params(ctx); A.lambda_dev = SC(lambda);
    A.threshold = threshold; A.run_start = ctx->run_start.as<unsigned>(); A.run_end = ctx->run_end.as<unsigned>();
    A.pos_data = ctx->pos_data; A.sv_label = ctx->sv_label.as<unsigned>(); A.mlog = ctx->ML; A.log_cap = std::max(1u, ctx->S);
    A.ctl = SC(mctl); A.S_cap = p.S_cap; A.E_cap = p.E_cap; A.resume = resume ? 1 : 0;
    A.big = nullptr; A.big_cursor = nullptr;
    if (big) {
        const size_t bb = (FastSmem::big_bytes(p.S_cap, p.E_cap) + 255) & ~(size_t)255;
        F3PS_CUDA_OK(ctx->lean_big.ensure(bb + lean_cursor_bytes(p.S_cap) + LeanWideScratch::bytes));
        A.big = (char*)ctx->lean_big.p; A.big_cursor = (unsigned*)((char*)ctx->lean_big.p + bb);
    }
    const size_t entries = 2 * (size_t)ctx->E + (big ? 8 : 1) * kLeanPoolSlack;     // (edge ids: 2 bytes, L2 variant 4)
    F3PS_CUDA_OK(ctx->adj_pool.ensure(entries * (big ? 4 : 2)));
    A.adj_pool = ctx->adj_pool.as<unsigned short>(); A.pool_cap = (unsigned)entries;
    A.trace = nullptr; A.trace_first = ctx->merge_trace_first;
    if (p.prof && !big) {
        F3PS_CUDA_OK(ctx->merge_trace.ensure(256 * 32 * 4));
        F3PS_CUDA_OK(cudaMemsetAsync(ctx->merge_trace.p, 0, 256 * 32 * 4, ctx->stream));
        A.trace = ctx->merge_trace.as<unsigned>();
    }
    return F3PS_OK;
}
int launch_resident(f3ps_ctx* ctx, const MergePlan& p, float threshold, bool resume) {
    FastArgs A;
    int rc = fast_args(ctx, p, threshold, resume, A); if (rc) return rc;
    void (*kern)(FastArgs) = p.kind == kMergeL2 ? (p.prof ? merge_fast_big_kernel<true> : merge_fast_big_kernel<false>)
                           : p.threads == kFastThreadsSolo ? (p.prof ? merge_fast_kernel<true, kFastThreadsSolo> : merge_fast_kernel<false, kFastThreadsSolo>)
                           : (p.prof ? merge_fast_kernel<true, kFastThreads> : merge_fast_kernel<false, kFastThreads>);
    rc = smem_opt_in(ctx, (const void*)kern, kSmemMax); if (rc) return rc;
    LAUNCH(ctx, kern, 1, p.threads, p.smem, A);
    return F3PS_OK;
}
// the general kernel (any graph) from the initial state; PK = one packed incidence word per edge (16 + 16 or 32 + 32 bits)
template <typename PK>
int launch_general(f3ps_ctx* ctx, float threshold) {
    const size_t Sc = std::max(1u, ctx->S), Ec = std::max(1u, ctx->E);
    const size_t per = (Ec * 4 + 255) & ~(size_t)255, per8 = (Ec * 8 + 255) & ~(size_t)255;
    unsigned n2 = 2048; while (n2 < Ec) n2 <<= 1;
    const size_t perS = (Sc * 4 + 255) & ~(size_t)255, sortb = (size_t)n2 * sizeof(MergeSortRec);
    F3PS_CUDA_OK(ctx->merge_scratch.ensure(6 * per + 2 * per8 + per + per8 + perS + sortb));
    char* sp = (char*)ctx->merge_scratch.p;
    MergeScratch scr;
    scr.st[0] = (long long*)sp; sp += per8; scr.st[1] = (long long*)sp; sp += per8;
    scr.sortbuf = (MergeSortRec*)sp; sp += sortb;
    scr.e[0] = (int*)sp; sp += per; scr.e[1] = (int*)sp; sp += per; scr.w[0] = (float*)sp; sp += per; scr.w[1] = (float*)sp; sp += per;
    scr.x[0] = (unsigned*)sp; sp += per; scr.x[1] = (unsigned*)sp; sp += per; scr.cls = (unsigned char*)sp; sp += per;
    scr.mark = (unsigned*)sp; sp += perS;
    const size_t dyn = (size_t)kMergeSortSmem * sizeof(MergeSortRec);
    int rc = smem_opt_in(ctx, (const void*)merge_kernel<PK>, dyn); if (rc) return rc;
    LAUNCH(ctx, merge_kernel<PK>, 1, kMergeThreads, dyn, ctx->R1, ctx->E1, SC(n_edges), SC(xctl.n_sv), edge_params(ctx), SC(lambda), threshold,
           ctx->run_start.as<unsigned>(), ctx->run_end.as<unsigned>(), ctx->order, ctx->gxyz, ctx->sv_label.as<unsigned>(), ctx->ML, (unsigned)Sc,
           SC(mctl), scr, (PK*)sp, ctx->pos_data);
    return F3PS_OK;
}
LabelArgs label_args(const f3ps_ctx* ctx) {
    LabelArgs A;
    A.R = ctx->R1; A.n_sv_ptr = SC(xctl.n_sv); A.run_start = ctx->run_start.as<unsigned>(); A.run_end = ctx->run_end.as<unsigned>();
    A.run_out_off = ctx->run_out_off.as<unsigned>(); A.run_dense = ctx->run_dense.as<unsigned>(); A.region_dense = ctx->region_dense.as<unsigned>();
    A.n_out = SC(n_out);
    A.pos_run = ctx->pos_run.as<unsigned>(); A.n_pos = ctx->n_pos; A.order = ctx->order; A.vox_xyz = ctx->gxyz;
    A.out_xyz = ctx->out_xyz.as<float>(); A.out_label = ctx->out_label.as<unsigned>(); A.out_voxel = ctx->out_voxel.as<unsigned>();
    A.vox_segment = ctx->vox_segment.as<unsigned>();
    A.pos_label = ctx->graph_from_host ? nullptr : ctx->sorted_label; A.owner = ctx->graph_from_host ? nullptr : ctx->owner0.as<unsigned>();
    A.scalars = (const unsigned*)ctx->d_sc;
    return A;
}
// after the replay's scalars reached the host; the merged state is one level, its threshold (f3ps_merge_levels records more)
int merge_done(f3ps_ctx* ctx, float threshold) {
    if (ctx->h_sc->mctl.error) return ctx_fail(ctx, F3PS_ERR_CAPACITY, "merge kernel reported an internal capacity error");
    ctx->n_out = ctx->h_sc->n_out;
    ctx->lv_thr.assign(1, threshold); ctx->lv_M = ctx->h_sc->mctl.n_merges;
    ctx->progress = P_MERGED;
    return F3PS_OK;
}

// stage mark i of every frame of a chunk, on the stream of its first frame (the lead), which runs the chunk's kernels
int mark_chunk(f3ps_ctx** ctxs, const std::vector<int>& chunk, int i) {
    f3ps_ctx* ctx = ctxs[chunk[0]];
    for (int f : chunk) { F3PS_CUDA_OK(cudaEventRecord(ctxs[f]->ev[i], ctx->stream)); ctxs[f]->ev_valid[i] = true; }
    return F3PS_OK;
}
// One round of a chunk on its lead's stream, without a host wait: the merge kernel (a grid whose CTA k replays frame k, or the
// frame's own kernel), then -- with supervoxels -- Clustering::get_labeled_cloud (dense segment ids, the labelled voxel cloud),
// then the scalars' read-back (a chunk of one copies its own; a grid gathers every frame's on the device for one copy).
int launch_chunk(f3ps_ctx** ctxs, const std::vector<int>& chunk, const std::vector<MergePlan>& step, const std::vector<char>& resume,
                 float threshold) {
    static thread_local FastBatch B;                         // 32 KB each: not on the stack
    static thread_local LabelBatch L;
    f3ps_ctx* ctx = ctxs[chunk[0]];
    const unsigned nf = (unsigned)chunk.size();
    int rc;
    if (ctx->S) {
        if (nf > 1) {
            size_t bytes = 0;                                // every frame brings its own table capacities (the layout is per CTA)
            for (unsigned k = 0; k < nf; ++k) {
                f3ps_ctx* m = ctxs[chunk[k]];
                rc = fast_args(m, step[chunk[k]], threshold, false, B.a[k]); if (rc) return rc;
                bytes = std::max(bytes, step[chunk[k]].smem);
                if (m->stream != ctx->stream) {              // the lead's stream runs the grid: it waits for everybody's set-up
                    F3PS_CUDA_OK(cudaEventRecord(m->ev_batch, m->stream));
                    F3PS_CUDA_OK(cudaStreamWaitEvent(ctx->stream, m->ev_batch, 0));
                }
            }
            rc = smem_opt_in(ctx, (const void*)merge_fast_batch_kernel, kSmemMax); if (rc) return rc;
            LAUNCH(ctx, merge_fast_batch_kernel, nf, kFastThreads, bytes, B);
        } else {
            const MergePlan& p = step[chunk[0]];
            rc = p.kind != kMergeGeneral ? launch_resident(ctx, p, threshold, resume[chunk[0]])
               : ctx->S < 65536u ? launch_general<unsigned>(ctx, threshold) : launch_general<unsigned long long>(ctx, threshold);
            if (rc) return rc;
        }
        rc = mark_chunk(ctxs, chunk, 10); if (rc) return rc;
        int gx = 1;
        for (unsigned k = 0; k < nf; ++k) {
            f3ps_ctx* m = ctxs[chunk[k]];
            m->merge_path = resume[chunk[k]] ? 6 : step[chunk[k]].kind;
            L.a[k] = label_args(m);
            gx = std::max(gx, grid_for(m->n_pos, 256));
        }
        LAUNCH(ctx, dense_label_batch_kernel, nf, 1024, 0, L);
        LAUNCH(ctx, labeled_cloud_batch_kernel, dim3(gx, nf), 256, 0, L);
    }
    rc = mark_chunk(ctxs, chunk, 8); if (rc) return rc;
    if (nf == 1) {
        F3PS_CUDA_OK(cudaMemcpyAsync(ctx->h_sc, ctx->d_sc, sizeof(DevScalars), cudaMemcpyDeviceToHost, ctx->stream));
        return F3PS_OK;
    }
    static_assert(sizeof(DevScalars) % 4 == 0, "DevScalars is gathered as words");
    F3PS_CUDA_OK(ctx->batch_sc.ensure(kFastBatchMax * sizeof(DevScalars)));
    if (!ctx->h_batch_sc) F3PS_CUDA_OK(cudaMallocHost(&ctx->h_batch_sc, kFastBatchMax * sizeof(DevScalars)));
    LAUNCH(ctx, scalars_gather_kernel, nf, 128, 0, L, (unsigned)(sizeof(DevScalars) / 4), ctx->batch_sc.as<unsigned>());
    F3PS_CUDA_OK(cudaMemcpyAsync(ctx->h_batch_sc, ctx->batch_sc.p, nf * sizeof(DevScalars), cudaMemcpyDeviceToHost, ctx->stream));
    return F3PS_OK;
}
// Clustering::cluster(threshold) of n handles on one device, graphs built: f3ps_merge (n = 1) and f3ps_merge_batch.
// The replay runs in rounds, one step per frame and round: a fresh replay from the frame's plan; a continuation on the L2 variant
// (merge_path 6) when the shared-memory variant stopped IN FRONT of a merge whose two adjacency lists hold more entries than it
// has worker threads (nothing of that merge has happened); or, after any other stop (adjacency pool or stamp range exhausted, a
// merge with more than 65,534 entries on the L2 variant), the general kernel replaying the whole sequence from the initial state.
// Fresh frames of the shared-memory kernel without phase counters share grids of at most kFastBatchMax frames: independent
// streams share at most 32 hardware queues, so at most 32 single-CTA merge kernels overlap, and a grid has no such cap.  Every
// other frame, one left alone in its chunk included, is a chunk of one that runs its plan's own kernel on its own stream.  The
// host waits only after every chunk of a round is in flight.
//
// No member stream waits for a grid: a stream parked behind a grid that runs for tens of milliseconds would hold its hardware
// queue, and the work other handles enqueue on that queue (the next group's front stages in a pipelined sweep) would wait for
// the grid too.  The call returns only after the host has seen every lead stream finish, so later work on a member's own stream
// (getters, levels, the next frame) needs no event wait.
int merge_frames(f3ps_ctx** ctxs, int n, float threshold) {
    std::vector<MergePlan> step(n);                          // each frame's kernel in the current round
    std::vector<char> resume(n, 0);                          // that kernel continues from the stopped state
    std::vector<int> grid, single;
    for (int i = 0; i < n; ++i) {
        f3ps_ctx* ctx = ctxs[i];
        int rc = merge_begin(ctx); if (rc) return rc;
        ctx->merge_path = 0;                                 // no supervoxels: no kernel runs (a reused handle must not report its last frame's)
        step[i] = plan_merge(ctx);
        if (ctx->S && (rc = mark(ctx, 9))) return rc;
        (ctx->S && step[i].kind == kMergeShared && !step[i].prof ? grid : single).push_back(i);
    }
    std::vector<std::vector<int>> chunks;
    for (size_t g0 = 0; g0 < grid.size(); g0 += kFastBatchMax)
        chunks.emplace_back(grid.begin() + g0, grid.begin() + std::min(grid.size(), g0 + (size_t)kFastBatchMax));
    for (int i : single) chunks.push_back({i});
    while (!chunks.empty()) {
        for (const auto& c : chunks) { int rc = launch_chunk(ctxs, c, step, resume, threshold); if (rc) return rc; }
        std::vector<std::vector<int>> next;
        for (const auto& c : chunks) {
            f3ps_ctx* lead = ctxs[c[0]];
            { f3ps_ctx* ctx = lead; F3PS_CUDA_OK(wait_stream(ctx)); }
            for (size_t k = 0; k < c.size(); ++k) {
                f3ps_ctx* ctx = ctxs[c[k]];
                MergePlan& p = step[c[k]];
                if (c.size() > 1) memcpy(ctx->h_sc, lead->h_batch_sc + k, sizeof(DevScalars));
                int rc;
                if (!ctx->h_sc->mctl.error || p.kind == kMergeGeneral) { if ((rc = merge_done(ctx, threshold))) return rc; continue; }
                resume[c[k]] = ctx->h_sc->mctl.error == kFastErrTouched && p.to_l2;
                if (resume[c[k]]) {
                    F3PS_CUDA_OK(cudaMemsetAsync(SC(mctl.error), 0, 4, ctx->stream));
                    p = plan_l2(ctx);
                } else {
                    if ((rc = merge_restart(ctx))) return rc;
                    p.kind = kMergeGeneral;
                }
                next.push_back({c[k]});
            }
        }
        chunks.swap(next);
    }
    return F3PS_OK;
}
}
}
int f3ps_merge(f3ps_ctx* ctx, float threshold) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    if (ctx->progress < P_EXPANDED)                            // std::logic_error of Clustering::cluster (src/clustering.cpp:671-673)
        return ctx_fail(ctx, F3PS_ERR_LOGIC, "Cannot call 'cluster' before setting an initial state with 'set_initialstate'");
    cudaSetDevice(ctx->device);
    if (ctx->progress < P_GRAPH) { int rc = f3ps_graph(ctx); if (rc) return rc; }   // if (!init_initial_weights) init_weights()  (:675-676)
    return merge_frames(&ctx, 1, threshold);
}

// Every handle must be on the same device; the results per handle are exactly those of f3ps_merge(handle, threshold).
int f3ps_merge_batch(f3ps_ctx** ctxs, int n, float threshold) {
    if (!ctxs || n < 1) return F3PS_ERR_INVALID_ARGUMENT;
    for (int i = 0; i < n; ++i) {
        if (!ctxs[i]) return F3PS_ERR_INVALID_ARGUMENT;
        if (ctxs[i]->device != ctxs[0]->device) return ctx_fail(ctxs[i], F3PS_ERR_INVALID_ARGUMENT, "f3ps_merge_batch: handles on different devices");
        if (ctxs[i]->progress < P_EXPANDED)
            return ctx_fail(ctxs[i], F3PS_ERR_LOGIC, "Cannot call 'cluster' before setting an initial state with 'set_initialstate'");
    }
    cudaSetDevice(ctxs[0]->device);
    for (int i = 0; i < n; ++i)
        if (ctxs[i]->progress < P_GRAPH) { int rc = f3ps_graph(ctxs[i]); if (rc) return rc; }
    return merge_frames(ctxs, n, threshold);
}

// ctas_per_frame = 0: K5's cooperative grid covers the whole GPU (lowest latency for a single frame, the default);
// ctas_per_frame > 0 caps it at that many CTAs.  max_concurrent must be 0.
int f3ps_set_expand_sharing(f3ps_ctx* ctx, int ctas_per_frame, int max_concurrent) {
    if (!ctx || ctas_per_frame < 0 || ctas_per_frame > 2 * kSMs || max_concurrent != 0) return F3PS_ERR_INVALID_ARGUMENT;
    ctx->expand_ctas = ctas_per_frame;
    return F3PS_OK;
}

int f3ps_set_expand_kernel(f3ps_ctx* ctx, int which, int cluster_ctas) {
    if (!ctx || which < 0 || which > 2 || cluster_ctas < 0 || cluster_ctas > kExpandClusterMax) return F3PS_ERR_INVALID_ARGUMENT;
    ctx->expand_kernel_choice = which;
    ctx->expand_cluster_ctas = cluster_ctas;
    return F3PS_OK;
}

int f3ps_set_blocking_wait(f3ps_ctx* ctx, int blocking) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    ctx->blocking_wait = blocking != 0;
    return F3PS_OK;
}

int f3ps_set_merge_kernel(f3ps_ctx* ctx, int which) {
    if (!ctx || which < 0 || which > 5 || which == 1) return F3PS_ERR_INVALID_ARGUMENT;
    ctx->merge_kernel_choice = which;
    return F3PS_OK;
}

int f3ps_extract(f3ps_ctx* ctx) {
    int rc;
    if ((rc = f3ps_voxelize(ctx))) return rc;
    if ((rc = f3ps_neighbors(ctx))) return rc;
    if ((rc = f3ps_normals(ctx))) return rc;
    if ((rc = f3ps_seeds(ctx))) return rc;
    if ((rc = f3ps_expand(ctx))) return rc;
    return f3ps_graph(ctx);
}
int f3ps_run(f3ps_ctx* ctx, float threshold) {
    int rc = f3ps_extract(ctx);
    if (rc) return rc;
    return f3ps_merge(ctx, threshold);
}


// =====================================================================================================
// Slab mode (SURVEY.md section 8e row 2; BASELINE config 5): one cloud, one slab of the x-major Morton key space per
// GPU.  The per-rank pieces live here, the splitter rule and the assembly of the replicated voxel table included; the host
// drivers (f3ps/slab.py, host/slab_host.cpp) issue only the exchanges between them on this handle's stream: all-reduce of
// the bounding box and the key histogram, all-to-all of the points, all-gather of the voxel slices and the normal slices.
// From f3ps_seeds on, every rank runs the ordinary stages on the whole table.
extern "C++" {
namespace {
template <typename KeyT>
int slab_keys_typed(f3ps_ctx* ctx, PointLoader pl, int shift, unsigned bins, unsigned* d_hist) {
    const int64_t N = ctx->n_points;
    F3PS_CUDA_OK(ctx->keys_a.ensure(N * sizeof(KeyT))); F3PS_CUDA_OK(ctx->keys_b.ensure(N * sizeof(KeyT)));
    F3PS_CUDA_OK(ctx->vals_a.ensure(N * 4)); F3PS_CUDA_OK(ctx->vals_b.ensure(N * 4));
    KeygenOp<KeyT> kop{pl, ctx->vp.use_transform, SC(fp), ctx->keys_a.as<KeyT>(), ctx->vals_a.as<unsigned>()};
    int rc = run_compact(ctx, kop, nullptr, N, SC(n_valid)); if (rc) return rc;
    LAUNCH(ctx, slab_key_hist_kernel<KeyT>, grid_for(N, 256 * 4, kSMs * 8), 256, 0, ctx->keys_a.as<KeyT>(), SC(n_valid), shift, bins, d_hist);
    return F3PS_OK;
}
template <typename KeyT>
int slab_route_typed(f3ps_ctx* ctx, PointLoader pl, const SlabSplitters& sp, int world, float4* d_send) {
    const int64_t N = ctx->n_points;
    F3PS_CUDA_OK(ctx->slab_dest.ensure(N * 4)); F3PS_CUDA_OK(ctx->starts.ensure((N + 1) * 4));
    LAUNCH(ctx, slab_dest_kernel<KeyT>, grid_for(N, 256 * 4, kSMs * 8), 256, 0, ctx->keys_a.as<KeyT>(), SC(n_valid), sp,
           ctx->slab_dest.as<unsigned>(), ctx->slab_tot.as<unsigned>());
    unsigned* sk; unsigned* sv;        // stable: input order survives inside a destination
    int rc = sort_pairs<unsigned>(ctx, ctx->slab_dest.as<unsigned>(), ctx->vals_a.as<unsigned>(), ctx->starts.as<unsigned>(), ctx->vals_b.as<unsigned>(),
                                  ctx->slab_dest.as<unsigned>(), ctx->vals_a.as<unsigned>(), SC(n_valid), N, bits_for((unsigned)std::max(1, world - 1)), &sk, &sv);
    if (rc) return rc;
    LAUNCH(ctx, slab_pack_kernel, grid_for(N, 256 * 2, kSMs * 8), 256, 0, pl, sv, SC(n_valid), d_send);
    return F3PS_OK;
}
} // namespace
} // extern "C++"

int f3ps_slab_reset(f3ps_ctx* ctx) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    ctx->slab_frame = false; ctx->slab_range = false;
    ctx->progress = std::min(ctx->progress, (int)P_INPUT);
    return F3PS_OK;
}

// bounding box of this rank's points (transformed space): d_box8 = ord_min[3], ord_max[3], any_finite, 0 in the
// order-preserving unsigned encoding (all-reduce MIN / MAX / MAX as unsigned)
int f3ps_slab_bbox(f3ps_ctx* ctx, uint32_t* d_box8) {
    if (!ctx || !d_box8) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_INPUT, "f3ps_slab_bbox"); if (rc) return rc;
    cudaSetDevice(ctx->device);
    DevScalars init; memset(&init, 0, sizeof init);
    for (int a = 0; a < 3; ++a) { init.fp.ord_min[a] = 0xffffffffu; init.fp.ord_max[a] = 0u; }
    *ctx->h_sc = init;
    F3PS_CUDA_OK(cudaMemcpyAsync(ctx->d_sc, ctx->h_sc, sizeof(DevScalars), cudaMemcpyHostToDevice, ctx->stream));
    PointLoader pl{ctx->d_points, ctx->stride, ctx->vp.fold_negative_z};
    if (ctx->n_points > 0)
        LAUNCH(ctx, bbox_kernel, grid_for(ctx->n_points, 256 * 4, kSMs * 8), 256, 0, pl, ctx->n_points, ctx->vp.use_transform, SC(fp));
    F3PS_CUDA_OK(cudaMemcpyAsync(d_box8, SC(fp.ord_min), 24, cudaMemcpyDeviceToDevice, ctx->stream));
    F3PS_CUDA_OK(cudaMemcpyAsync(d_box8 + 6, SC(fp.any_finite), 4, cudaMemcpyDeviceToDevice, ctx->stream));
    F3PS_CUDA_OK(cudaMemsetAsync(d_box8 + 7, 0, 4, ctx->stream));
    ctx->slab_frame = false;
    return F3PS_OK;
}

// the reduced box of the whole cloud -> OctreePointCloud::defineBoundingBox / getKeyBitSize, identical on every rank
int f3ps_slab_set_frame(f3ps_ctx* ctx, const uint32_t* d_box8) {
    if (!ctx || !d_box8) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_INPUT, "f3ps_slab_set_frame"); if (rc) return rc;
    cudaSetDevice(ctx->device);
    F3PS_CUDA_OK(cudaMemcpyAsync(SC(fp.ord_min), d_box8, 24, cudaMemcpyDeviceToDevice, ctx->stream));
    F3PS_CUDA_OK(cudaMemcpyAsync(SC(fp.any_finite), d_box8 + 6, 4, cudaMemcpyDeviceToDevice, ctx->stream));
    LAUNCH(ctx, frame_setup_kernel, 1, 1, 0, SC(fp), ctx->vp.voxel_res);
    rc = pull_scalars(ctx); if (rc) return rc;
    ctx->slab_fp = ctx->h_sc->fp; ctx->slab_frame = true; ctx->slab_bits = 0;
    ctx->depth = ctx->slab_fp.depth;
    if (ctx->depth > 21) return ctx_fail(ctx, F3PS_ERR_CAPACITY, "adjacency octree depth > 21");
    ctx->key64 = 3 * ctx->depth > 32;
    return F3PS_OK;
}

// Morton keys of this rank's valid points + histogram of their top `top_bits` bits (d_hist: 1 << top_bits counters, device).
// The handle keeps the binning for f3ps_slab_route: bin = key >> shift, min(top_bits, 3 * depth) bits
int f3ps_slab_keys(f3ps_ctx* ctx, int top_bits, uint32_t* d_hist) {
    if (!ctx || !d_hist || top_bits < 1 || top_bits > kSlabHistBitsMax) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_INPUT, "f3ps_slab_keys"); if (rc) return rc;
    if (!ctx->slab_frame) return ctx_fail(ctx, F3PS_ERR_LOGIC, "f3ps_slab_keys: f3ps_slab_set_frame has not run");
    cudaSetDevice(ctx->device);
    const int kb = 3 * ctx->depth, tb = std::min(top_bits, std::max(1, kb)), shift = std::max(0, kb - tb);
    ctx->slab_bits = tb; ctx->slab_shift = shift;
    F3PS_CUDA_OK(cudaMemsetAsync(d_hist, 0, (size_t)4 << top_bits, ctx->stream));
    PointLoader pl{ctx->d_points, ctx->stride, ctx->vp.fold_negative_z};
    if (ctx->n_points == 0) { F3PS_CUDA_OK(cudaMemsetAsync(SC(n_valid), 0, 4, ctx->stream)); return F3PS_OK; }
    return ctx->key64 ? slab_keys_typed<uint64_t>(ctx, pl, shift, 1u << tb, d_hist) : slab_keys_typed<uint32_t>(ctx, pl, shift, 1u << tb, d_hist);
}

// Equal-count cuts of the key space: cut r is the first bin boundary at or after r/world of the points, never below the cut
// before it, shifted to a Morton key.  out[world - 1] ascend; rank r owns [out[r-1], out[r]).  Host only: no CUDA call.
int f3ps_slab_choose_splitters(const uint32_t* hist, int n_bins, int world, int shift, uint64_t* out) {
    if (!hist || n_bins < 1 || world < 1 || shift < 0 || shift > 63 || !out) return F3PS_ERR_INVALID_ARGUMENT;
    std::vector<uint64_t> cum((size_t)n_bins);
    uint64_t total = 0;
    for (int i = 0; i < n_bins; ++i) cum[(size_t)i] = total += hist[i];
    uint64_t prev = 0;
    for (int r = 1; r < world; ++r) {
        const uint64_t target = total * (uint64_t)r / (uint64_t)world;
        uint64_t b = (uint64_t)(std::lower_bound(cum.begin(), cum.end(), target) - cum.begin()) + 1;
        b = prev = std::min<uint64_t>(std::max(b, prev), (uint64_t)n_bins);
        out[r - 1] = b << shift;
    }
    return F3PS_OK;
}

// d_hist: the histogram of f3ps_slab_keys, all-reduced over the ranks (device; may be NULL when world == 1).  Cuts the key space
// with f3ps_slab_choose_splitters and packs this rank's valid points as 16-byte records {x, y, z, rgba} into d_send (capacity:
// n points), grouped by destination rank, input order kept inside a group; counts[world] = records per destination.
int f3ps_slab_route(f3ps_ctx* ctx, int world, const uint32_t* d_hist, void* d_send, int64_t* counts) {
    if (!ctx || world < 1 || world > kSlabMaxWorld || (world > 1 && !d_hist) || !counts) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_INPUT, "f3ps_slab_route"); if (rc) return rc;
    if (!ctx->slab_frame || !ctx->slab_bits) return ctx_fail(ctx, F3PS_ERR_LOGIC, "f3ps_slab_route: f3ps_slab_set_frame / f3ps_slab_keys have not run");
    cudaSetDevice(ctx->device);
    for (int r = 0; r < world; ++r) counts[r] = 0;
    if (ctx->n_points == 0) return F3PS_OK;
    SlabSplitters sp; memset(&sp, 0, sizeof sp); sp.n = world - 1;
    if (world > 1) {
        std::vector<uint32_t> hist((size_t)1 << ctx->slab_bits);
        F3PS_CUDA_OK(cudaMemcpyAsync(hist.data(), d_hist, hist.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
        F3PS_CUDA_OK(wait_stream(ctx));
        uint64_t cut[kSlabMaxWorld];
        rc = f3ps_slab_choose_splitters(hist.data(), (int)hist.size(), world, ctx->slab_shift, cut); if (rc) return rc;
        for (int r = 0; r + 1 < world; ++r) { sp.key[r] = cut[r]; if (r && cut[r] < cut[r - 1]) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "splitters must ascend"); }
    }
    F3PS_CUDA_OK(ctx->slab_tot.ensure(kSlabMaxWorld * 4));
    F3PS_CUDA_OK(cudaMemsetAsync(ctx->slab_tot.p, 0, kSlabMaxWorld * 4, ctx->stream));
    PointLoader pl{ctx->d_points, ctx->stride, ctx->vp.fold_negative_z};
    rc = ctx->key64 ? slab_route_typed<uint64_t>(ctx, pl, sp, world, (float4*)d_send) : slab_route_typed<uint32_t>(ctx, pl, sp, world, (float4*)d_send);
    if (rc) return rc;
    unsigned tot[kSlabMaxWorld];
    F3PS_CUDA_OK(cudaMemcpyAsync(tot, ctx->slab_tot.p, sizeof tot, cudaMemcpyDeviceToHost, ctx->stream));
    F3PS_CUDA_OK(wait_stream(ctx));
    for (int r = 0; r < world; ++r) counts[r] = tot[r];
    return F3PS_OK;
}

// device arrays the driver exchanges in place (pointer, elements, bytes per element)
int f3ps_slab_array(f3ps_ctx* ctx, int which, void** ptr, int64_t* n, int* elem_bytes) {
    if (!ctx || !ptr || !n || !elem_bytes) return F3PS_ERR_INVALID_ARGUMENT;
    const int64_t V = ctx->V;
    switch (which) {
    case F3PS_SLAB_VOX_XYZ: *ptr = ctx->vox_xyz.p; *n = V; *elem_bytes = 16; break;
    case F3PS_SLAB_VOX_RGB: *ptr = ctx->vox_rgb.p; *n = V; *elem_bytes = 16; break;
    case F3PS_SLAB_VOX_KEY: *ptr = ctx->vox_key.p; *n = V; *elem_bytes = 8; break;
    case F3PS_SLAB_VOX_NORMAL: *ptr = ctx->vox_normal.p; *n = V; *elem_bytes = 16; break;
    case F3PS_SLAB_VOX_CURV: *ptr = ctx->vox_curv.p; *n = V; *elem_bytes = 4; break;
    default: return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "unknown slab array");
    }
    return F3PS_OK;
}

// Right after f3ps_voxelize on the received points (ctx->V = this rank's v_local voxels): the voxel tables grow to the WHOLE
// cloud's n_voxels, this rank's slice moves to [own_begin, own_begin + v_local), the slice it computes from here on.  The caller
// then fills the other ranks' slices in place (f3ps_slab_array) before f3ps_neighbors.
int f3ps_slab_set_voxels(f3ps_ctx* ctx, int64_t n_voxels, int64_t own_begin) {
    if (!ctx || n_voxels < 0 || own_begin < 0) return F3PS_ERR_INVALID_ARGUMENT;
    if (n_voxels >= (1ll << 30)) return ctx_fail(ctx, F3PS_ERR_CAPACITY, "more than 2^30 voxels");
    if (!ctx->slab_frame) return ctx_fail(ctx, F3PS_ERR_LOGIC, "f3ps_slab_set_voxels: f3ps_slab_set_frame has not run");
    if (ctx->progress != P_VOXELS || ctx->slab_range) return ctx_fail(ctx, F3PS_ERR_LOGIC, "f3ps_slab_set_voxels: must follow f3ps_voxelize");
    const size_t v_local = ctx->V, V = (size_t)n_voxels, Vc = std::max<size_t>(1, V), at = (size_t)own_begin;
    if (at + v_local > V) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "f3ps_slab_set_voxels: own_begin + this rank's voxels > n_voxels");
    cudaSetDevice(ctx->device);
    f3ps::DevBuf* tab[3] = {&ctx->vox_xyz, &ctx->vox_rgb, &ctx->vox_key};
    const size_t eb[3] = {16, 16, 8}, off[3] = {0, 16, 32};          // bytes per voxel; the slice's place in the spare buffer
    bool move = at != 0;
    for (int i = 0; i < 3; ++i) move = move || tab[i]->cap < Vc * eb[i];
    if (move) {        // through the spare buffer: growing a table frees its contents, and the slice's two places may overlap
        F3PS_CUDA_OK(ctx->slab_spare.ensure(std::max<size_t>(1, v_local) * 40));
        char* spare = ctx->slab_spare.as<char>();
        for (int i = 0; i < 3 && v_local; ++i)
            F3PS_CUDA_OK(cudaMemcpyAsync(spare + off[i] * v_local, tab[i]->p, v_local * eb[i], cudaMemcpyDeviceToDevice, ctx->stream));
        F3PS_CUDA_OK(wait_stream(ctx));
        for (int i = 0; i < 3; ++i) {
            F3PS_CUDA_OK(tab[i]->ensure(Vc * eb[i]));
            if (v_local) F3PS_CUDA_OK(cudaMemcpyAsync(tab[i]->as<char>() + at * eb[i], spare + off[i] * v_local, v_local * eb[i], cudaMemcpyDeviceToDevice, ctx->stream));
        }
    }
    ctx->V = (unsigned)V;
    const unsigned v32 = (unsigned)V;
    F3PS_CUDA_OK(cudaMemcpyAsync(SC(n_voxels), &v32, 4, cudaMemcpyHostToDevice, ctx->stream));
    F3PS_CUDA_OK(wait_stream(ctx));
    ctx->own_begin = (unsigned)at; ctx->own_end = (unsigned)(at + v_local); ctx->slab_range = true;
    ctx->progress = P_VOXELS;
    return mark(ctx, 1);
}

int f3ps_merge_profile(f3ps_ctx* ctx, uint64_t cycles[32]) {
    if (!ctx || !cycles) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_MERGED, "f3ps_merge_profile"); if (rc) return rc;
    for (int i = 0; i < 32; ++i) cycles[i] = ctx->h_sc->mctl.phase_cycles[i];
    return F3PS_OK;
}

int f3ps_merge_trace(f3ps_ctx* ctx, int64_t first_merge, uint32_t* out, int64_t capacity_words) {
    if (!ctx || first_merge < 0) return F3PS_ERR_INVALID_ARGUMENT;
    ctx->merge_trace_first = (unsigned)first_merge;          // takes effect at the next f3ps_merge with kernel choice 4
    if (!out) return F3PS_OK;
    if (capacity_words < 256 * 32 || !ctx->merge_trace.p) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "f3ps_merge_trace: no trace recorded or buffer below 8192 words");
    cudaSetDevice(ctx->device);
    F3PS_CUDA_OK(cudaMemcpyAsync(out, ctx->merge_trace.p, 256 * 32 * 4, cudaMemcpyDeviceToHost, ctx->stream));
    F3PS_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    return F3PS_OK;
}

int f3ps_expand_profile(f3ps_ctx* ctx, uint64_t ns[8]) {
    if (!ctx || !ns) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_EXPANDED, "f3ps_expand_profile"); if (rc) return rc;
    if ((rc = pull_scalars(ctx))) return rc;
    for (int i = 0; i < 8; ++i) ns[i] = ctx->h_sc->xctl.t_phase[i];
    return F3PS_OK;
}

int f3ps_stage_ms(f3ps_ctx* ctx, int stage, float* ms) {
    if (!ctx || !ms || stage < 0 || stage > 8) return F3PS_ERR_INVALID_ARGUMENT;
    cudaSetDevice(ctx->device);
    F3PS_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    int i0, i1;
    if (stage == F3PS_STAGE_TOTAL) { i0 = 0; i1 = 8; }
    else if (stage == F3PS_STAGE_MERGE_KERNEL) { i0 = 9; i1 = 10; }
    else if (stage == F3PS_STAGE_MERGE) { i0 = 7; i1 = 8; }
    else { i0 = stage; i1 = stage + 1; }
    if (!ctx->ev_valid[i0] || !ctx->ev_valid[i1]) return ctx_fail(ctx, F3PS_ERR_LOGIC, "stage has not run");
    F3PS_CUDA_OK(cudaEventElapsedTime(ms, ctx->ev[i0], ctx->ev[i1]));
    return F3PS_OK;
}

} // extern "C"

// =====================================================================================================
// results
namespace {
int d2h(f3ps_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (!bytes || !dst) return F3PS_OK;
    F3PS_CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return F3PS_OK;
}
int fin(f3ps_ctx* ctx) { F3PS_CUDA_OK(wait_stream(ctx)); return F3PS_OK; }
int cap_check(f3ps_ctx* ctx, int64_t need_n, int64_t capacity) {
    if (capacity < need_n) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "output capacity too small");
    return F3PS_OK;
}
}

extern "C" {

int f3ps_get_counts(f3ps_ctx* ctx, f3ps_counts* out) {
    if (!ctx || !out) return F3PS_ERR_INVALID_ARGUMENT;
    cudaSetDevice(ctx->device);
    int rc = pull_scalars(ctx); if (rc) return rc;
    const DevScalars& h = *ctx->h_sc;
    memset(out, 0, sizeof *out);
    out->n_points = ctx->n_points; out->n_valid = ctx->n_valid; out->n_voxels = ctx->V; out->depth = ctx->depth;
    out->seed_depth = h.sb.depth; out->n_seed_cells = (int)ctx->n_cells; out->n_seeds = (int)ctx->S0;
    out->n_supervoxels = (int)ctx->S; out->n_edges = (int)ctx->E;
    out->n_merges = (int)h.mctl.n_merges; out->n_segments = (int)h.mctl.regions_alive; out->n_edges_left = (int)h.mctl.edges_alive;
    out->rounds = ctx->rounds; out->sweeps = (int)h.xctl.sweeps_total; out->n_labeled = (int)ctx->n_out;
    out->lambda = h.lambda;
    out->max_touched = (int)h.mctl.max_touched; out->fold_steps = (int64_t)h.mctl.fold_steps;
    out->nan_weights = (int)(h.mctl.nan_weights + h.nan_weights_init);
    out->merge_path = ctx->merge_path;
    if (ctx->progress < P_MERGED) { out->n_segments = (int)ctx->S; out->n_edges_left = (int)ctx->E; }
    return F3PS_OK;
}

int f3ps_get_voxel_keys(f3ps_ctx* ctx, uint32_t* keys, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_VOXELS, "f3ps_get_voxel_keys"); if (rc) return rc;
    if ((rc = cap_check(ctx, ctx->V, capacity))) return rc;
    std::vector<uint64_t> m(ctx->V);
    if ((rc = d2h(ctx, m.data(), ctx->vox_key.p, (size_t)ctx->V * 8))) return rc;
    if ((rc = fin(ctx))) return rc;
    for (unsigned v = 0; v < ctx->V; ++v) morton_decode(m[v], keys[3 * v], keys[3 * v + 1], keys[3 * v + 2]);
    return F3PS_OK;
}

int f3ps_get_voxel_centroids(f3ps_ctx* ctx, float* xyz, float* rgb, uint32_t* rgba, int32_t* count, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_VOXELS, "f3ps_get_voxel_centroids"); if (rc) return rc;
    if ((rc = cap_check(ctx, ctx->V, capacity))) return rc;
    const unsigned V = ctx->V;
    std::vector<float4> a(V), b(V);
    if ((rc = d2h(ctx, a.data(), ctx->vox_xyz.p, (size_t)V * 16))) return rc;
    if ((rc = d2h(ctx, b.data(), ctx->vox_rgb.p, (size_t)V * 16))) return rc;
    if ((rc = fin(ctx))) return rc;
    for (unsigned v = 0; v < V; ++v) {
        if (xyz) { xyz[3 * v] = a[v].x; xyz[3 * v + 1] = a[v].y; xyz[3 * v + 2] = a[v].z; }
        if (rgb) { rgb[3 * v] = b[v].x; rgb[3 * v + 1] = b[v].y; rgb[3 * v + 2] = b[v].z; }
        if (rgba) memcpy(&rgba[v], &a[v].w, 4);
        if (count) count[v] = (int)b[v].w;
    }
    return F3PS_OK;
}

int f3ps_get_point_voxel(f3ps_ctx* ctx, int32_t* pv, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_VOXELS, "f3ps_get_point_voxel"); if (rc) return rc;
    if ((rc = cap_check(ctx, ctx->n_points, capacity))) return rc;
    if ((rc = d2h(ctx, pv, ctx->point_voxel.p, (size_t)ctx->n_points * 4))) return rc;
    return fin(ctx);
}

int f3ps_get_voxel_neighbors(f3ps_ctx* ctx, int32_t* nbr, int32_t* nbr_count, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_NEIGHBORS, "f3ps_get_voxel_neighbors"); if (rc) return rc;
    if ((rc = cap_check(ctx, ctx->V, capacity))) return rc;
    const unsigned V = ctx->V;
    std::vector<int> rows((size_t)V * kNbrStride);
    if ((rc = d2h(ctx, rows.data(), ctx->nbr_row.p, rows.size() * 4))) return rc;
    if ((rc = fin(ctx))) return rc;
    for (unsigned v = 0; v < V; ++v) {
        if (nbr) for (int r = 0; r < 27; ++r) nbr[(size_t)v * 27 + r] = rows[(size_t)v * kNbrStride + r];
        if (nbr_count) nbr_count[v] = rows[(size_t)v * kNbrStride + 27];
    }
    return F3PS_OK;
}

int f3ps_get_voxel_normals(f3ps_ctx* ctx, float* normal4, float* curvature, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_NORMALS, "f3ps_get_voxel_normals"); if (rc) return rc;
    if ((rc = cap_check(ctx, ctx->V, capacity))) return rc;
    if ((rc = d2h(ctx, normal4, ctx->vox_normal.p, (size_t)ctx->V * 16))) return rc;
    if ((rc = d2h(ctx, curvature, ctx->vox_curv.p, (size_t)ctx->V * 4))) return rc;
    return fin(ctx);
}

int f3ps_get_seeds(f3ps_ctx* ctx, int32_t* seed_voxel, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_SEEDS, "f3ps_get_seeds"); if (rc) return rc;
    if ((rc = cap_check(ctx, ctx->S0, capacity))) return rc;
    if ((rc = d2h(ctx, seed_voxel, ctx->seeds.p, (size_t)ctx->S0 * 4))) return rc;
    return fin(ctx);
}

int f3ps_get_voxel_labels(f3ps_ctx* ctx, uint32_t* label, float* distance, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_EXPANDED, "f3ps_get_voxel_labels"); if (rc) return rc;
    if (ctx->graph_from_host) return ctx_fail(ctx, F3PS_ERR_LOGIC, "no voxel labels: graph was supplied by the caller");
    if ((rc = cap_check(ctx, ctx->V, capacity))) return rc;
    if ((rc = d2h(ctx, label, ctx->owner0.p, (size_t)ctx->V * 4))) return rc;
    if ((rc = d2h(ctx, distance, ctx->dist0.p, (size_t)ctx->V * 4))) return rc;
    return fin(ctx);
}

int f3ps_get_supervoxels(f3ps_ctx* ctx, uint32_t* label, float* centroid, float* mean_rgb, float* normal4, int32_t* n_voxels, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_EXPANDED, "f3ps_get_supervoxels"); if (rc) return rc;
    if (ctx->graph_from_host) return ctx_fail(ctx, F3PS_ERR_LOGIC, "supervoxels were supplied by the caller");
    if ((rc = cap_check(ctx, ctx->S, capacity))) return rc;
    const unsigned S = ctx->S, Sc = ctx->S0 + 2;
    std::vector<unsigned> lab(S);
    std::vector<float4> x(Sc), c(Sc), n(Sc);
    if ((rc = d2h(ctx, lab.data(), ctx->sv_label.p, (size_t)S * 4))) return rc;
    if ((rc = d2h(ctx, x.data(), ctx->cen_xyz.p, (size_t)Sc * 16))) return rc;
    if ((rc = d2h(ctx, c.data(), ctx->cen_rgb.p, (size_t)Sc * 16))) return rc;
    if ((rc = d2h(ctx, n.data(), ctx->cen_nrm.p, (size_t)Sc * 16))) return rc;
    if ((rc = fin(ctx))) return rc;
    for (unsigned s = 0; s < S; ++s) {
        const unsigned l = lab[s];
        if (label) label[s] = l;
        if (centroid) { centroid[3 * s] = x[l].x; centroid[3 * s + 1] = x[l].y; centroid[3 * s + 2] = x[l].z; }
        if (mean_rgb) { mean_rgb[3 * s] = c[l].x; mean_rgb[3 * s + 1] = c[l].y; mean_rgb[3 * s + 2] = c[l].z; }
        if (normal4) { normal4[4 * s] = n[l].x; normal4[4 * s + 1] = n[l].y; normal4[4 * s + 2] = n[l].z; normal4[4 * s + 3] = n[l].w; }
        if (n_voxels) n_voxels[s] = (int)x[l].w;
    }
    return F3PS_OK;
}

int f3ps_get_supervoxel_voxels(f3ps_ctx* ctx, int32_t* voxel_index, int64_t* offsets, int64_t cap_voxels, int64_t cap_sv) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_GRAPH, "f3ps_get_supervoxel_voxels"); if (rc) return rc;
    const unsigned S = ctx->S, P = ctx->n_pos;
    if ((rc = cap_check(ctx, S, cap_sv))) return rc;
    std::vector<unsigned> rs(S), re(S), ord(P);
    if ((rc = d2h(ctx, rs.data(), ctx->run_start.p, (size_t)S * 4))) return rc;
    if ((rc = d2h(ctx, re.data(), ctx->run_end.p, (size_t)S * 4))) return rc;
    if ((rc = d2h(ctx, ord.data(), ctx->order, (size_t)P * 4))) return rc;
    if ((rc = fin(ctx))) return rc;
    int64_t tot = 0;
    for (unsigned s = 0; s < S; ++s) tot += re[s] - rs[s];
    if ((rc = cap_check(ctx, tot, cap_voxels))) return rc;
    int64_t o = 0;
    for (unsigned s = 0; s < S; ++s) {
        if (offsets) offsets[s] = o;
        for (unsigned i = rs[s]; i < re[s]; ++i) { if (voxel_index) voxel_index[o] = (int)ord[i]; ++o; }
    }
    if (offsets) offsets[S] = o;
    return F3PS_OK;
}

static int fetch_edges(f3ps_ctx* ctx, const EdgeArrays& EA, unsigned n, std::vector<unsigned>& a, std::vector<unsigned>& b, std::vector<float>& dc,
                       std::vector<float>& dg, std::vector<float>& w, std::vector<long long>& st, std::vector<unsigned>& lab) {
    a.resize(n); b.resize(n); dc.resize(n); dg.resize(n); w.resize(n); st.resize(n); lab.resize(ctx->S);
    int rc;
    if ((rc = d2h(ctx, a.data(), EA.a, (size_t)n * 4))) return rc;
    if ((rc = d2h(ctx, b.data(), EA.b, (size_t)n * 4))) return rc;
    if ((rc = d2h(ctx, dc.data(), EA.dc, (size_t)n * 4))) return rc;
    if ((rc = d2h(ctx, dg.data(), EA.dg, (size_t)n * 4))) return rc;
    if ((rc = d2h(ctx, w.data(), EA.w, (size_t)n * 4))) return rc;
    if ((rc = d2h(ctx, st.data(), EA.stamp, (size_t)n * 8))) return rc;
    if ((rc = d2h(ctx, lab.data(), ctx->sv_label.p, (size_t)ctx->S * 4))) return rc;
    return fin(ctx);
}

int f3ps_get_edges(f3ps_ctx* ctx, uint32_t* ab, float* delta_c, float* delta_g, float* weight, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_GRAPH, "f3ps_get_edges"); if (rc) return rc;
    if ((rc = cap_check(ctx, ctx->E, capacity))) return rc;
    std::vector<unsigned> a, b, lab; std::vector<float> dc, dg, w; std::vector<long long> st;
    if ((rc = fetch_edges(ctx, ctx->E0, ctx->E, a, b, dc, dg, w, st, lab))) return rc;
    for (unsigned e = 0; e < ctx->E; ++e) {
        if (ab) { ab[2 * e] = lab[a[e]]; ab[2 * e + 1] = lab[b[e]]; }
        if (delta_c) delta_c[e] = dc[e];
        if (delta_g) delta_g[e] = dg[e];
        if (weight) weight[e] = w[e];
    }
    return F3PS_OK;
}

int f3ps_get_adjacency(f3ps_ctx* ctx, uint32_t* pairs, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_GRAPH, "f3ps_get_adjacency"); if (rc) return rc;
    if ((rc = cap_check(ctx, 2 * (int64_t)ctx->E, capacity))) return rc;
    std::vector<unsigned> a, b, lab; std::vector<float> dc, dg, w; std::vector<long long> st;
    if ((rc = fetch_edges(ctx, ctx->E0, ctx->E, a, b, dc, dg, w, st, lab))) return rc;
    std::vector<std::pair<unsigned, unsigned>> p;
    for (unsigned e = 0; e < ctx->E; ++e) { p.push_back({lab[a[e]], lab[b[e]]}); p.push_back({lab[b[e]], lab[a[e]]}); }
    std::sort(p.begin(), p.end());
    for (size_t i = 0; i < p.size(); ++i) { pairs[2 * i] = p[i].first; pairs[2 * i + 1] = p[i].second; }
    return F3PS_OK;
}

int f3ps_get_cdf(f3ps_ctx* ctx, float* cdf_c, float* cdf_g, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_GRAPH, "f3ps_get_cdf"); if (rc) return rc;
    if (ctx->mp.merge_mode != F3PS_EQUALIZATION) return ctx_fail(ctx, F3PS_ERR_LOGIC, "no CDF unless the merging criterion is EQUALIZATION");
    if ((rc = cap_check(ctx, ctx->mp.bins, capacity))) return rc;
    if ((rc = d2h(ctx, cdf_c, ctx->cdf_c.p, (size_t)ctx->mp.bins * 4))) return rc;
    if ((rc = d2h(ctx, cdf_g, ctx->cdf_g.p, (size_t)ctx->mp.bins * 4))) return rc;
    return fin(ctx);
}

int f3ps_get_merge_log(f3ps_ctx* ctx, uint32_t* ab, float* weight, uint32_t* left, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_MERGED, "f3ps_get_merge_log"); if (rc) return rc;
    const unsigned M = ctx->h_sc->mctl.n_merges;
    if ((rc = cap_check(ctx, M, capacity))) return rc;
    std::vector<unsigned> a(M), b(M), el(M), rl(M);
    if ((rc = d2h(ctx, a.data(), ctx->ML.a, (size_t)M * 4))) return rc;
    if ((rc = d2h(ctx, b.data(), ctx->ML.b, (size_t)M * 4))) return rc;
    if ((rc = d2h(ctx, el.data(), ctx->ML.edges_left, (size_t)M * 4))) return rc;
    if ((rc = d2h(ctx, rl.data(), ctx->ML.regions_left, (size_t)M * 4))) return rc;
    if ((rc = d2h(ctx, weight, ctx->ML.w, (size_t)M * 4))) return rc;
    if ((rc = fin(ctx))) return rc;
    for (unsigned m = 0; m < M; ++m) {
        if (ab) { ab[2 * m] = a[m]; ab[2 * m + 1] = b[m]; }
        if (left) { left[2 * m] = el[m]; left[2 * m + 1] = rl[m]; }
    }
    return F3PS_OK;
}

int f3ps_get_state_regions(f3ps_ctx* ctx, uint32_t* label, float* centroid, float* normal, int32_t* n_voxels, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_GRAPH, "f3ps_get_state_regions"); if (rc) return rc;
    const RegionArrays& R = ctx->progress >= P_MERGED ? ctx->R1 : ctx->R0;
    const unsigned S = ctx->S;
    std::vector<int> n(S); std::vector<float4> c(S), nn(S); std::vector<unsigned> lab(S);
    if ((rc = d2h(ctx, n.data(), R.n, (size_t)S * 4))) return rc;
    if ((rc = d2h(ctx, c.data(), R.centroid, (size_t)S * 16))) return rc;
    if ((rc = d2h(ctx, nn.data(), R.normal, (size_t)S * 16))) return rc;
    if ((rc = d2h(ctx, lab.data(), ctx->sv_label.p, (size_t)S * 4))) return rc;
    if ((rc = fin(ctx))) return rc;
    int64_t k = 0;
    for (unsigned s = 0; s < S; ++s) if (n[s] > 0) ++k;
    if ((rc = cap_check(ctx, k, capacity))) return rc;
    k = 0;
    for (unsigned s = 0; s < S; ++s) {
        if (n[s] <= 0) continue;
        if (label) label[k] = lab[s];
        if (centroid) { centroid[3 * k] = c[s].x; centroid[3 * k + 1] = c[s].y; centroid[3 * k + 2] = c[s].z; }
        if (normal) { normal[3 * k] = nn[s].x; normal[3 * k + 1] = nn[s].y; normal[3 * k + 2] = nn[s].z; }
        if (n_voxels) n_voxels[k] = n[s];
        ++k;
    }
    return F3PS_OK;
}

int f3ps_get_region_mean_color(f3ps_ctx* ctx, int32_t rank, float rgb[3]) {
    if (!ctx || !rgb) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_GRAPH, "f3ps_get_region_mean_color"); if (rc) return rc;
    if (rank < 0 || (unsigned)rank >= ctx->S) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "region rank out of range");
    float4 m;
    if ((rc = d2h(ctx, &m, ctx->R0.mean + rank, 16))) return rc;
    if ((rc = fin(ctx))) return rc;
    rgb[0] = m.y; rgb[1] = m.z; rgb[2] = m.w;
    return F3PS_OK;
}

int f3ps_get_state_edges(f3ps_ctx* ctx, uint32_t* ab, float* weight, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_GRAPH, "f3ps_get_state_edges"); if (rc) return rc;
    const EdgeArrays& EA = ctx->progress >= P_MERGED ? ctx->E1 : ctx->E0;
    std::vector<unsigned> a, b, lab; std::vector<float> dc, dg, w; std::vector<long long> st;
    if ((rc = fetch_edges(ctx, EA, ctx->E, a, b, dc, dg, w, st, lab))) return rc;
    std::vector<unsigned> idx;
    for (unsigned e = 0; e < ctx->E; ++e) if (st[e] != kDeadStamp) idx.push_back(e);
    if ((rc = cap_check(ctx, (int64_t)idx.size(), capacity))) return rc;
    std::sort(idx.begin(), idx.end(), [&](unsigned x, unsigned y) { return w[x] < w[y] || (w[x] == w[y] && st[x] < st[y]); });   // multimap order
    for (size_t i = 0; i < idx.size(); ++i) {
        const unsigned e = idx[i];
        if (ab) { ab[2 * i] = lab[a[e]]; ab[2 * i + 1] = lab[b[e]]; }
        if (weight) weight[i] = w[e];
    }
    return F3PS_OK;
}

int f3ps_get_labeled_cloud(f3ps_ctx* ctx, float* xyz, uint32_t* label, uint32_t* voxel_index, int64_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_MERGED, "f3ps_get_labeled_cloud"); if (rc) return rc;
    if ((rc = cap_check(ctx, ctx->n_out, capacity))) return rc;
    if ((rc = d2h(ctx, xyz, ctx->out_xyz.p, (size_t)ctx->n_out * 12))) return rc;
    if ((rc = d2h(ctx, label, ctx->out_label.p, (size_t)ctx->n_out * 4))) return rc;
    if ((rc = d2h(ctx, voxel_index, ctx->out_voxel.p, (size_t)ctx->n_out * 4))) return rc;
    return fin(ctx);
}

int f3ps_get_voxel_segments_device(f3ps_ctx* ctx, const uint32_t** device_ptr, int64_t* n) {
    if (!ctx || !device_ptr || !n) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_MERGED, "f3ps_get_voxel_segments_device"); if (rc) return rc;
    *device_ptr = ctx->vox_segment.as<uint32_t>(); *n = ctx->n_pos;
    return F3PS_OK;
}

// ---- segmentation levels (kernels_levels.cuh) ---------------------------------------------------------
extern "C++" {
namespace {
// merge forest of the last replay: parent and merge time per initial supervoxel
int levels_forest(f3ps_ctx* ctx) {
    const unsigned S = ctx->S, M = ctx->lv_M;
    const size_t Sc = std::max(1u, S);
    F3PS_CUDA_OK(ctx->lv_parent.ensure(Sc * 4)); F3PS_CUDA_OK(ctx->lv_when.ensure(Sc * 4));
    F3PS_CUDA_OK(cudaMemsetAsync(ctx->lv_when.p, 0xff, Sc * 4, ctx->stream));
    if (M) LAUNCH(ctx, levels_forest_kernel, grid_for(M, 256), 256, 0, ctx->ML.a, ctx->ML.b, M, ctx->sv_label.as<unsigned>(), S,
                  ctx->lv_parent.as<unsigned>(), ctx->lv_when.as<unsigned>());
    return F3PS_OK;
}
// lv_small = thresholds, merges and segment counts of up to kMaxLevels levels
unsigned* levels_m(f3ps_ctx* ctx) { return ctx->lv_small.as<unsigned>() + kMaxLevels; }
unsigned* levels_nseg(f3ps_ctx* ctx) { return ctx->lv_small.as<unsigned>() + 2 * kMaxLevels; }
// merges, segment counts and per-supervoxel labels (lv_seg[S][level_row(L)]) of L ascending thresholds, on the forest
int levels_tables(f3ps_ctx* ctx, const float* thr, int L) {
    const unsigned S = ctx->S; const int Lp = level_row(L);
    const size_t Sc = std::max(1u, S);
    F3PS_CUDA_OK(ctx->lv_small.ensure(3 * kMaxLevels * 4));
    F3PS_CUDA_OK(ctx->lv_dense.ensure((size_t)L * Sc * 4)); F3PS_CUDA_OK(ctx->lv_seg.ensure((size_t)Lp * Sc * 4));
    F3PS_CUDA_OK(cudaMemcpyAsync(ctx->lv_small.p, thr, (size_t)L * 4, cudaMemcpyHostToDevice, ctx->stream));
    LAUNCH(ctx, levels_prefix_kernel, 1, 1024, 2 * L * 4, ctx->ML.w, ctx->lv_M, ctx->lv_small.as<float>(), L, levels_m(ctx));
    LAUNCH(ctx, levels_dense_kernel, L, 1024, 0, ctx->lv_when.as<unsigned>(), S, levels_m(ctx), ctx->lv_dense.as<unsigned>(), levels_nseg(ctx));
    if (S) LAUNCH(ctx, levels_roots_kernel, grid_for(S, 256), 256, 0, ctx->lv_parent.as<unsigned>(), ctx->lv_when.as<unsigned>(), levels_m(ctx),
                  ctx->lv_dense.as<unsigned>(), S, L, Lp, ctx->lv_seg.as<unsigned>());
    return F3PS_OK;
}
// the level tables of the handle's levels, built on first use after a merge; voxels: the voxel table [V][level_row(L)] as well
int levels_ready(f3ps_ctx* ctx, bool voxels, const char* what) {
    int rc = need(ctx, P_MERGED, what); if (rc) return rc;
    if (ctx->lv_thr.empty()) return ctx_fail(ctx, F3PS_ERR_LOGIC, std::string(what) + ": no merged state");
    cudaSetDevice(ctx->device);
    const int L = (int)ctx->lv_thr.size(), Lp = level_row(L);
    if (ctx->lv_built < 1) {
        if ((rc = levels_forest(ctx)) || (rc = levels_tables(ctx, ctx->lv_thr.data(), L))) return rc;
        ctx->lv_m_h.clear(); ctx->lv_nseg_h.clear();
        ctx->lv_built = 1;
    }
    if (voxels && ctx->lv_built < 2) {
        const unsigned V = ctx->V, P = ctx->n_pos;
        F3PS_CUDA_OK(ctx->lv_vox.ensure(std::max<size_t>(1, (size_t)V * Lp) * 4));
        F3PS_CUDA_OK(cudaMemsetAsync(ctx->lv_vox.p, 0xff, (size_t)V * Lp * 4, ctx->stream));
        const bool host = ctx->graph_from_host;
        if (P) LAUNCH(ctx, levels_voxel_kernel, grid_for(P, 256), 256, 0, ctx->pos_run.as<unsigned>(), P, host ? ctx->graph_vox.as<unsigned>() : ctx->order,
                      host ? nullptr : ctx->sorted_label, host ? nullptr : ctx->owner0.as<unsigned>(), ctx->lv_seg.as<unsigned>(), Lp, ctx->lv_vox.as<unsigned>());
        ctx->lv_built = 2;
    }
    return F3PS_OK;
}
// labels[L][n] = voxel table row pv[i] (pv == nullptr: row i).  Device memory: one launch, enqueued.  Host memory: through a
// staging buffer of at most kLevelStageWords words, a chunk of points at a time (a 50 M-point cloud at 41 levels would
// otherwise hold 8 GB of device memory for a copy).
constexpr size_t kLevelStageWords = (size_t)1 << 24;
int level_labels(f3ps_ctx* ctx, const int* pv, int64_t n, uint32_t* labels, int64_t capacity, int on_device) {
    const int L = (int)ctx->lv_thr.size(), Lp = level_row(L);
    const size_t words = (size_t)L * (size_t)n;
    int rc = cap_check(ctx, (int64_t)words, capacity); if (rc) return rc;
    if (!words) return F3PS_OK;
    if (!labels) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "no output buffer");
    const unsigned* table = ctx->lv_vox.as<unsigned>();
    if (on_device) {
        const int vec = ((uintptr_t)labels % 16 == 0 && n % 4 == 0) ? 1 : 0;
        LAUNCH(ctx, level_point_labels_kernel, grid_for((n + 3) / 4, 256), 256, 0, pv, 0, (long long)n, table, L, Lp, (unsigned*)labels, vec);
        return F3PS_OK;
    }
    const int64_t chunk = std::min<int64_t>(n, std::max<int64_t>(4, (int64_t)(kLevelStageWords / L) & ~(int64_t)3));
    F3PS_CUDA_OK(ctx->lv_points.ensure((size_t)chunk * L * 4));
    unsigned* stage = ctx->lv_points.as<unsigned>();
    for (int64_t p0 = 0; p0 < n; p0 += chunk) {
        const int64_t m = std::min(chunk, n - p0);
        LAUNCH(ctx, level_point_labels_kernel, grid_for((m + 3) / 4, 256), 256, 0, pv ? pv + p0 : nullptr, (int)p0, (long long)m, table, L, Lp,
               stage, m % 4 == 0 ? 1 : 0);
        F3PS_CUDA_OK(cudaMemcpy2DAsync(labels + p0, (size_t)n * 4, stage, (size_t)m * 4, (size_t)m * 4, (size_t)L, cudaMemcpyDeviceToHost, ctx->stream));
    }
    return fin(ctx);
}
// segment extraction (kernels_segments.cuh): the members of segments 0..K-1 of `level` grouped into g -- the points (pv =
// point_voxel over the n input points) or the n voxels (pv == nullptr) -- unless g already holds that level.  One wait, for the
// two sizes the host needs to size the sort (members, segments).
int segment_group(f3ps_ctx* ctx, int level, const int* pv, int64_t n, SegCsr& g) {
    if (g.level == level) return F3PS_OK;
    g.level = -1;
    const int Lp = level_row((int)ctx->lv_thr.size());
    const size_t nc = (size_t)std::max<int64_t>(n, 1), Sc = (size_t)ctx->S + 1;     // K <= S
    F3PS_CUDA_OK(g.keys_a.ensure(nc * 4)); F3PS_CUDA_OK(g.keys_b.ensure(nc * 4));
    F3PS_CUDA_OK(g.vals_a.ensure(nc * 4)); F3PS_CUDA_OK(g.vals_b.ensure(nc * 4));
    F3PS_CUDA_OK(g.counts.ensure((Sc + 1) * 4)); F3PS_CUDA_OK(g.offsets.ensure(Sc * 12));
    unsigned* sizes = g.counts.as<unsigned>();              // [0] members, [1] segments, then the K counts
    SegmentKeyOp op{pv, ctx->lv_vox.as<unsigned>(), Lp, level, g.keys_a.as<unsigned>(), g.vals_a.as<unsigned>()};
    int rc = run_compact(ctx, op, nullptr, n, sizes); if (rc) return rc;
    F3PS_CUDA_OK(cudaMemcpyAsync(sizes + 1, levels_nseg(ctx) + level, 4, cudaMemcpyDeviceToDevice, ctx->stream));
    unsigned h[2];
    if ((rc = d2h(ctx, h, sizes, sizeof h)) || (rc = fin(ctx))) return rc;
    g.n = h[0]; g.K = h[1];
    unsigned* counts = sizes + 2;
    const unsigned* keys = g.keys_a.as<unsigned>();
    g.index = g.vals_a.as<unsigned>();
    if (g.K > 1 && g.n > 1) {                                // one segment: the compaction's index order is the grouping
        unsigned *sk, *sv;
        rc = sort_pairs<unsigned>(ctx, g.keys_a.as<unsigned>(), g.vals_a.as<unsigned>(), g.keys_b.as<unsigned>(), g.vals_b.as<unsigned>(),
                                  g.keys_a.as<unsigned>(), g.vals_a.as<unsigned>(), nullptr, g.n, bits_for(g.K - 1), &sk, &sv);
        if (rc) return rc;
        keys = sk; g.index = sv;
    }
    if (g.K) F3PS_CUDA_OK(cudaMemsetAsync(counts, 0, (size_t)g.K * 4, ctx->stream));
    if (g.n) LAUNCH(ctx, segment_count_kernel, grid_for((g.n + kSegRun - 1) / kSegRun, 256), 256, 0, keys, sizes, counts);
    LAUNCH(ctx, segment_offsets_kernel, 1, 1024, 0, counts, g.K, g.off(), g.chunk_off());
    g.level = level;
    return F3PS_OK;
}
// checks shared by the segment getters; points: the getter needs the handle's input cloud
int segments_ready(f3ps_ctx* ctx, int level, bool points, const char* what) {
    if (points && ctx->graph_from_host) return ctx_fail(ctx, F3PS_ERR_LOGIC, std::string(what) + ": no input cloud, the graph was supplied by the caller");
    if (points && ctx->slab_range) return ctx_fail(ctx, F3PS_ERR_LOGIC, std::string(what) + ": slab mode, the handle holds no input cloud of its own voxels");
    int rc = levels_ready(ctx, true, what); if (rc) return rc;
    if (level < 0 || level >= (int)ctx->lv_thr.size()) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, std::string(what) + ": level out of range");
    return F3PS_OK;
}
// offsets[K+1] and index[n] of g into caller memory: enqueued (device) or copied and waited for (host)
int segment_copy(f3ps_ctx* ctx, const SegCsr& g, int64_t* offsets, int32_t* index, int32_t cap_segments, int64_t cap_index, int on_device) {
    int rc;
    if ((rc = cap_check(ctx, (int64_t)g.K + 1, cap_segments)) || (rc = cap_check(ctx, g.n, cap_index))) return rc;
    if (!offsets || (g.n && !index)) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "no output buffer");
    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    F3PS_CUDA_OK(cudaMemcpyAsync(offsets, g.off(), ((size_t)g.K + 1) * 8, kind, ctx->stream));
    if (g.n) F3PS_CUDA_OK(cudaMemcpyAsync(index, g.index, (size_t)g.n * 4, kind, ctx->stream));
    return on_device ? F3PS_OK : fin(ctx);
}
} // namespace
} // extern "C++"

int f3ps_merge_levels(f3ps_ctx* ctx, const float* thresholds, int n_levels) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    if (!thresholds || n_levels < 1 || n_levels > kMaxLevels) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "f3ps_merge_levels: 1 to 256 thresholds");
    for (int k = 0; k < n_levels; ++k)
        if (!std::isfinite(thresholds[k]) || (k && thresholds[k] < thresholds[k - 1]))
            return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "f3ps_merge_levels: thresholds must be finite and non-decreasing");
    int rc = f3ps_merge(ctx, thresholds[n_levels - 1]); if (rc) return rc;     // ONE replay; every level is a prefix of it
    ctx->lv_thr.assign(thresholds, thresholds + n_levels);
    return F3PS_OK;
}

int f3ps_get_levels(f3ps_ctx* ctx, int32_t* n_levels, float* thresholds, int32_t* n_merges, int32_t* n_segments, int32_t capacity) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = levels_ready(ctx, false, "f3ps_get_levels"); if (rc) return rc;
    const int L = (int)ctx->lv_thr.size();
    if (n_levels) *n_levels = L;
    if (!thresholds && !n_merges && !n_segments) return F3PS_OK;
    if ((rc = cap_check(ctx, L, capacity))) return rc;
    if ((n_merges || n_segments) && ctx->lv_m_h.empty()) {
        ctx->lv_m_h.resize(L); ctx->lv_nseg_h.resize(L);
        if ((rc = d2h(ctx, ctx->lv_m_h.data(), levels_m(ctx), (size_t)L * 4)) || (rc = d2h(ctx, ctx->lv_nseg_h.data(), levels_nseg(ctx), (size_t)L * 4)) ||
            (rc = fin(ctx))) { ctx->lv_m_h.clear(); return rc; }
    }
    for (int k = 0; k < L; ++k) {
        if (thresholds) thresholds[k] = ctx->lv_thr[k];
        if (n_merges) n_merges[k] = ctx->lv_m_h[k];
        if (n_segments) n_segments[k] = ctx->lv_nseg_h[k];
    }
    return F3PS_OK;
}

int f3ps_get_level_voxel_labels(f3ps_ctx* ctx, uint32_t* labels, int64_t capacity, int on_device) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = levels_ready(ctx, true, "f3ps_get_level_voxel_labels"); if (rc) return rc;
    return level_labels(ctx, nullptr, ctx->V, labels, capacity, on_device);
}

int f3ps_get_level_point_labels(f3ps_ctx* ctx, uint32_t* labels, int64_t capacity, int on_device) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    if (ctx->graph_from_host) return ctx_fail(ctx, F3PS_ERR_LOGIC, "f3ps_get_level_point_labels: no input cloud, the graph was supplied by the caller");
    if (ctx->slab_range) return ctx_fail(ctx, F3PS_ERR_LOGIC, "f3ps_get_level_point_labels: slab mode, the handle holds no input cloud of its own voxels");
    int rc = levels_ready(ctx, true, "f3ps_get_level_point_labels"); if (rc) return rc;
    return level_labels(ctx, ctx->point_voxel.as<int>(), ctx->n_points, labels, capacity, on_device);
}

int f3ps_get_segment_points(f3ps_ctx* ctx, int level, int64_t* offsets, int32_t* point_index, int32_t capacity_segments, int64_t capacity_points,
                            int on_device) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = segments_ready(ctx, level, true, "f3ps_get_segment_points"); if (rc) return rc;
    if ((rc = segment_group(ctx, level, ctx->point_voxel.as<int>(), ctx->n_points, ctx->seg_points))) return rc;
    return segment_copy(ctx, ctx->seg_points, offsets, point_index, capacity_segments, capacity_points, on_device);
}

int f3ps_get_segment_voxels(f3ps_ctx* ctx, int level, int64_t* offsets, int32_t* voxel_index, int32_t capacity_segments, int64_t capacity_voxels,
                            int on_device) {
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = segments_ready(ctx, level, false, "f3ps_get_segment_voxels"); if (rc) return rc;
    if ((rc = segment_group(ctx, level, nullptr, ctx->V, ctx->seg_voxels))) return rc;
    return segment_copy(ctx, ctx->seg_voxels, offsets, voxel_index, capacity_segments, capacity_voxels, on_device);
}

int f3ps_get_segment_info(f3ps_ctx* ctx, int level, f3ps_segment_info* out, int32_t capacity) {
    static_assert(sizeof(f3ps_segment_info) == 64, "f3ps_segment_info is 64 bytes");
    if (!ctx) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = segments_ready(ctx, level, true, "f3ps_get_segment_info"); if (rc) return rc;
    if ((rc = segment_group(ctx, level, ctx->point_voxel.as<int>(), ctx->n_points, ctx->seg_points)) ||
        (rc = segment_group(ctx, level, nullptr, ctx->V, ctx->seg_voxels))) return rc;
    const SegCsr& g = ctx->seg_points;
    const unsigned K = g.K;
    if ((rc = cap_check(ctx, K, capacity))) return rc;
    if (!K) return F3PS_OK;
    if (!out) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "no output buffer");
    const size_t chunks = ((size_t)g.n + kSegChunk - 1) / kSegChunk + K;     // >= the partials of all segments
    F3PS_CUDA_OK(ctx->seg_part.ensure(chunks * sizeof(SegPartial))); F3PS_CUDA_OK(ctx->seg_info.ensure((size_t)K * sizeof(f3ps_segment_info)));
    f3ps_segment_info* info = ctx->seg_info.as<f3ps_segment_info>();
    PointLoader pl{ctx->d_points, ctx->stride, ctx->vp.fold_negative_z};
    if (g.n) LAUNCH(ctx, segment_partials_kernel, (int)chunks, kSegThreads, 0, pl, g.index, g.off(), g.chunk_off(), K, ctx->seg_part.as<SegPartial>());
    LAUNCH(ctx, segment_info_kernel, (int)(((size_t)K * 32 + 255) / 256), 256, 0, ctx->seg_part.as<SegPartial>(), g.chunk_off(), g.off(),
           ctx->seg_voxels.off(), K, info);
    if (ctx->S) LAUNCH(ctx, segment_region_kernel, grid_for(ctx->S, 256), 256, 0, ctx->lv_dense.as<unsigned>() + (size_t)level * ctx->S,
                       ctx->sv_label.as<unsigned>(), ctx->S, info);
    if ((rc = d2h(ctx, out, info, (size_t)K * sizeof(f3ps_segment_info)))) return rc;
    return fin(ctx);
}

// ---- device self tests ------------------------------------------------------------------------------
// =====================================================================================================
// "next" row f1: Clustering::all_thresh (src/clustering.cpp:691-729) + Testing::eval_performance (src/testing.cpp:239-362).
extern "C++" {
namespace {
// Testing::compute_intersections' best matches + the seven scores, in the reference's float order.
// table[n_seg][n_truth] = inter_matrix; g[j] = truth segment sizes; N = truth->size().
f3ps_performance testing_scores(const std::vector<unsigned>& table, unsigned n_seg, unsigned n_truth, const std::vector<size_t>& g, size_t N) {
    // table has n_truth + 1 columns: the last one counts segmentation points without a ground-truth point at the same xyz
    auto inter = [&](unsigned i, unsigned j) -> size_t { return table[(size_t)i * (n_truth + 1) + j]; };
    std::vector<size_t> ssz(n_seg, 0);
    for (unsigned i = 0; i < n_seg; ++i) for (unsigned j = 0; j <= n_truth; ++j) ssz[i] += inter(i, j);
    // t_sizes: std::map<size_t, uint32_t>, insert keeps the FIRST truth segment of every size (testing.cpp:97-110)
    std::map<size_t, unsigned> t_sizes;
    if (n_seg) for (unsigned j = 0; j < n_truth; ++j) t_sizes.insert(std::make_pair(g[j], j));
    std::vector<long long> matches(n_truth, -1);
    for (auto it = t_sizes.rbegin(); it != t_sizes.rend(); ++it) {           // largest truth segment first (:112-137)
        const unsigned j = it->second;
        std::vector<size_t> col(n_seg);
        for (unsigned i = 0; i < n_seg; ++i) col[i] = inter(i, j);
        auto argmax = [&]() { long long r = 0; for (unsigned i = 1; i < n_seg; ++i) if (col[i] > col[(size_t)r]) r = i; return r; };   // Eigen maxCoeff: first maximum
        long long row = argmax();
        auto taken = [&](long long r) { for (long long m : matches) if (m == r) return true; return false; };
        while (taken(row)) {
            col[(size_t)row] = 0;
            bool any = false; for (size_t c : col) any = any || c != 0;
            if (any) row = argmax(); else { row = -1; break; }
        }
        matches[j] = row;
    }
    f3ps_performance pf;
    const float n = (float)N;
    {   // eval_voi (:305-335)
        float h_s = 0, h_t = 0, mi = 0;
        for (unsigned i = 0; i < n_seg; ++i) {
            const float p = (float)ssz[i];
            h_s -= std::log(p / n) * p / n;
            for (unsigned j = 0; j < n_truth; ++j) {
                const float q = (float)g[j];
                if (i == 0) h_t -= std::log(q / n) * q / n;
                const float r = (float)inter(i, j);
                if (r != 0) mi += std::log(((n * r) / (p * q))) * r / n;
            }
        }
        pf.voi = h_s + h_t - 2 * mi;
    }
    {   // eval_precision (:239-268)
        float p = 0, r = 0, fp = 0, fn = 0;
        for (unsigned j = 0; j < n_truth; ++j) {
            const long long i = matches[j];
            if (i != -1) {
                const float in = (float)inter((unsigned)i, j), sz = (float)ssz[(size_t)i], gg = (float)g[j];
                p += in * gg / sz; r += in; fp += (sz - in); fn += (gg - in);
            } else fn += (float)g[j];
        }
        pf.precision = p / n; pf.recall = r / n; pf.fpr = fp / n; pf.fnr = fn / n;
    }
    if (pf.precision == 0 && pf.recall == 0) pf.fscore = 0;                 // eval_fscore (:287-299)
    else pf.fscore = 2 * (pf.precision * pf.recall) / (pf.precision + pf.recall);
    {   // eval_wov (:342-357): count_union of two point sets = |s| + |t| - |s ^ t|
        float w = 0;
        for (unsigned j = 0; j < n_truth; ++j) {
            const long long i = matches[j];
            if (i != -1) {
                const float in = (float)inter((unsigned)i, j);
                const float un = (float)(ssz[(size_t)i] + g[j] - inter((unsigned)i, j));
                w += in * (float)g[j] / un;
            }
        }
        pf.wov = w / n;
    }
    return pf;
}
} // namespace
} // extern "C++"

int f3ps_eval_thresholds(f3ps_ctx* ctx, const uint32_t* truth_label, int64_t n_voxels, const uint32_t* extra_truth_label, int64_t n_extra,
                         const float* thresholds, int n_thresholds, f3ps_performance* perf, int32_t* n_segments, int32_t* n_merges_at) {
    if (!ctx || !truth_label || !thresholds || !perf || n_thresholds < 1 || n_extra < 0 || (n_extra > 0 && !extra_truth_label)) return F3PS_ERR_INVALID_ARGUMENT;
    int rc = need(ctx, P_GRAPH, "f3ps_eval_thresholds"); if (rc) return rc;
    if (n_voxels != (int64_t)ctx->V) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "one ground-truth label per voxel is required");
    for (int k = 1; k < n_thresholds; ++k) if (!(thresholds[k] >= thresholds[k - 1])) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "thresholds must ascend");
    cudaSetDevice(ctx->device);
    rc = f3ps_merge(ctx, thresholds[n_thresholds - 1]); if (rc) return rc;      // ONE replay; every threshold is a prefix of it
    const unsigned S = ctx->S, V = ctx->V, P = ctx->n_pos;
    if (ctx->n_out == 0) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "The pointcloud to be set as 'segm' cannot be empty");  // testing.cpp:413-416
    // Testing::label_map on the truth: dense labels in ascending label order, segment sizes
    std::map<unsigned, unsigned> tmap;
    size_t n_truth_points = 0;
    for (int64_t v = 0; v < n_voxels; ++v) if (truth_label[v] != 0xffffffffu) { tmap[truth_label[v]] = 0; ++n_truth_points; }
    for (int64_t v = 0; v < n_extra; ++v) { tmap[extra_truth_label[v]] = 0; ++n_truth_points; }
    if (n_truth_points == 0) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "The pointcloud to be set as 'truth' cannot be empty");
    unsigned Kt = 0; for (auto& kv : tmap) kv.second = Kt++;
    std::vector<unsigned> tdense((size_t)V); std::vector<size_t> g(Kt, 0);
    for (unsigned v = 0; v < V; ++v) {
        if (truth_label[v] == 0xffffffffu) { tdense[v] = Kt; continue; }     // no ground-truth point at this voxel's xyz
        tdense[v] = tmap[truth_label[v]]; g[tdense[v]]++;
    }
    for (int64_t v = 0; v < n_extra; ++v) g[tmap[extra_truth_label[v]]]++;    // truth points outside the segmentation's voxels
    const unsigned Kc = Kt + 1;
    if ((size_t)S * Kc > ((size_t)1 << 28)) return ctx_fail(ctx, F3PS_ERR_CAPACITY, "contingency table above 2^28 cells");
    F3PS_CUDA_OK(ctx->ev_truth.ensure((size_t)V * 4)); F3PS_CUDA_OK(ctx->ev_table.ensure(std::max<size_t>(1, (size_t)S * Kc) * 4));
    F3PS_CUDA_OK(cudaMemcpyAsync(ctx->ev_truth.p, tdense.data(), (size_t)V * 4, cudaMemcpyHostToDevice, ctx->stream));
    // the segmentation at every threshold: the level tables of the replay, kMaxLevels thresholds at a time
    rc = levels_forest(ctx); if (rc) return rc;
    std::vector<unsigned> table, m_at(kMaxLevels), nseg_at(kMaxLevels);
    unsigned m_prev = 0xffffffffu;
    for (int k0 = 0; k0 < n_thresholds; k0 += kMaxLevels) {
        const int L = std::min(kMaxLevels, n_thresholds - k0);
        rc = levels_tables(ctx, thresholds + k0, L); if (rc) return rc;
        if ((rc = d2h(ctx, m_at.data(), levels_m(ctx), (size_t)L * 4)) || (rc = d2h(ctx, nseg_at.data(), levels_nseg(ctx), (size_t)L * 4))) return rc;
        if ((rc = fin(ctx))) return rc;
        for (int j = 0; j < L; ++j) {
            const int k = k0 + j;
            const unsigned m = m_at[j];                                           // first step whose head weight is >= t (strict <, :388-389)
            if (n_merges_at) n_merges_at[k] = (int32_t)m;
            if (m == m_prev) { perf[k] = perf[k - 1]; if (n_segments) n_segments[k] = n_segments[k - 1]; continue; }
            m_prev = m;
            const unsigned n_seg = nseg_at[j];
            F3PS_CUDA_OK(cudaMemsetAsync(ctx->ev_table.p, 0, std::max<size_t>(1, (size_t)S * Kc) * 4, ctx->stream));
            if (P) LAUNCH(ctx, eval_table_kernel, grid_for(P, 256), 256, 0, ctx->pos_run.as<unsigned>(), ctx->order, P, ctx->lv_seg.as<unsigned>(),
                          level_row(L), j, ctx->ev_truth.as<unsigned>(), Kc, ctx->ev_table.as<unsigned>());
            table.resize((size_t)n_seg * Kc);
            if (n_seg) { if ((rc = d2h(ctx, table.data(), ctx->ev_table.p, (size_t)n_seg * Kc * 4))) return rc; if ((rc = fin(ctx))) return rc; }
            perf[k] = testing_scores(table, n_seg, Kt, g, n_truth_points);
            if (n_segments) n_segments[k] = (int32_t)n_seg;
        }
    }
    return F3PS_OK;      // the level tables now hold the sweep's thresholds: the handle's one level, the last, is rebuilt on demand
}


int f3ps_eval_label_pairs(f3ps_ctx* ctx, const uint32_t* seg, const uint32_t* truth, int64_t n_pairs, int32_t n_seg, int32_t n_truth,
                          const uint64_t* truth_sizes, int64_t n_truth_points, f3ps_performance* perf) {
    if (!ctx || !perf || n_pairs < 0 || n_seg < 0 || n_truth < 0 || (n_pairs > 0 && (!seg || !truth)) || (n_truth > 0 && !truth_sizes)) return F3PS_ERR_INVALID_ARGUMENT;
    if (n_pairs == 0) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "The pointcloud to be set as 'segm' cannot be empty");       // testing.cpp:413-416
    if (n_truth_points <= 0) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "The pointcloud to be set as 'truth' cannot be empty"); // :430-433
    for (int64_t i = 0; i < n_pairs; ++i)
        if (seg[i] >= (uint32_t)n_seg || truth[i] > (uint32_t)n_truth) return ctx_fail(ctx, F3PS_ERR_INVALID_ARGUMENT, "f3ps_eval_label_pairs: label out of range");
    const unsigned Kc = (unsigned)n_truth + 1u;
    if ((size_t)n_seg * Kc > ((size_t)1 << 28)) return ctx_fail(ctx, F3PS_ERR_CAPACITY, "contingency table above 2^28 cells");
    cudaSetDevice(ctx->device);
    const size_t cells = std::max<size_t>(1, (size_t)n_seg * Kc);
    F3PS_CUDA_OK(ctx->ev_dense.ensure((size_t)n_pairs * 4)); F3PS_CUDA_OK(ctx->ev_truth.ensure((size_t)n_pairs * 4)); F3PS_CUDA_OK(ctx->ev_table.ensure(cells * 4));
    F3PS_CUDA_OK(cudaMemcpyAsync(ctx->ev_dense.p, seg, (size_t)n_pairs * 4, cudaMemcpyHostToDevice, ctx->stream));
    F3PS_CUDA_OK(cudaMemcpyAsync(ctx->ev_truth.p, truth, (size_t)n_pairs * 4, cudaMemcpyHostToDevice, ctx->stream));
    F3PS_CUDA_OK(cudaMemsetAsync(ctx->ev_table.p, 0, cells * 4, ctx->stream));
    LAUNCH(ctx, eval_pairs_kernel, grid_for(n_pairs, 256), 256, 0, ctx->ev_dense.as<unsigned>(), ctx->ev_truth.as<unsigned>(), (long long)n_pairs, Kc, ctx->ev_table.as<unsigned>());
    std::vector<unsigned> table(cells);
    int rc = d2h(ctx, table.data(), ctx->ev_table.p, cells * 4); if (rc) return rc;
    if ((rc = fin(ctx))) return rc;
    std::vector<size_t> g((size_t)n_truth);
    for (int32_t j = 0; j < n_truth; ++j) g[(size_t)j] = (size_t)truth_sizes[j];
    *perf = testing_scores(table, (unsigned)n_seg, (unsigned)n_truth, g, (size_t)n_truth_points);
    return F3PS_OK;
}

static int test_map3(f3ps_ctx* ctx, int which, const float* in1, const float* in2, float* out, int64_t n) {
    if (!ctx || n < 0) return F3PS_ERR_INVALID_ARGUMENT;
    cudaSetDevice(ctx->device);
    DevBuf a, b, o;
    const size_t nb = (size_t)std::max<int64_t>(n, 1) * 12;
    int rc = F3PS_OK;
    do {
        if (a.ensure(nb) != cudaSuccess || b.ensure(nb) != cudaSuccess || o.ensure(nb) != cudaSuccess) { rc = ctx_fail(ctx, F3PS_ERR_CUDA, "cudaMalloc failed"); break; }
        cudaMemcpyAsync(a.p, in1, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream);
        if (in2) cudaMemcpyAsync(b.p, in2, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream);
        const int g = grid_for(n, 128);
        if (which == 0) lab_test_kernel<<<g, 128, 0, ctx->stream>>>(ctx->d_lab_lut, a.as<float>(), o.as<float>(), n);
        else if (which == 1) ciede_test_kernel<<<g, 128, 0, ctx->stream>>>(a.as<float>(), b.as<float>(), o.as<float>(), n);
        else rgb_eucl_test_kernel<<<g, 128, 0, ctx->stream>>>(a.as<float>(), b.as<float>(), o.as<float>(), n);
        ctx->launches++;
        cudaMemcpyAsync(out, o.p, (size_t)n * (which == 0 ? 12 : 4), cudaMemcpyDeviceToHost, ctx->stream);
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = ctx_fail_cuda(ctx, e, "self test", __FILE__, __LINE__);
    } while (0);
    a.release(); b.release(); o.release();
    return rc;
}
int f3ps_test_rgb2lab(f3ps_ctx* ctx, const float* rgb255, float* lab, int64_t n) { return test_map3(ctx, 0, rgb255, nullptr, lab, n); }
int f3ps_test_lab_ciede00(f3ps_ctx* ctx, const float* l1, const float* l2, float* out, int64_t n) { return test_map3(ctx, 1, l1, l2, out, n); }
int f3ps_test_rgb_eucl(f3ps_ctx* ctx, const float* c1, const float* c2, float* out, int64_t n) { return test_map3(ctx, 2, c1, c2, out, n); }

int f3ps_test_sort_pairs(f3ps_ctx* ctx, uint64_t* keys, uint32_t* values, int64_t n, int key_bits) {
    if (!ctx || n < 0 || key_bits < 1 || key_bits > 64) return F3PS_ERR_INVALID_ARGUMENT;
    cudaSetDevice(ctx->device);
    DevBuf ka, kb, va, vb;
    const size_t nk = (size_t)std::max<int64_t>(n, 1);
    int rc = F3PS_OK;
    do {
        if (ka.ensure(nk * 8) != cudaSuccess || kb.ensure(nk * 8) != cudaSuccess || va.ensure(nk * 4) != cudaSuccess || vb.ensure(nk * 4) != cudaSuccess) {
            rc = ctx_fail(ctx, F3PS_ERR_CUDA, "cudaMalloc failed"); break; }
        cudaMemcpyAsync(ka.p, keys, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(va.p, values, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream);
        unsigned long long* sk = ka.as<unsigned long long>(); unsigned* sv = va.as<unsigned>();
        if (n) {
            rc = sort_pairs<unsigned long long>(ctx, ka.as<unsigned long long>(), va.as<unsigned>(), kb.as<unsigned long long>(), vb.as<unsigned>(),
                                                ka.as<unsigned long long>(), va.as<unsigned>(), nullptr, n, key_bits, &sk, &sv);
            if (rc) break;
        }
        cudaMemcpyAsync(keys, sk, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream);
        cudaMemcpyAsync(values, sv, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream);
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = ctx_fail_cuda(ctx, e, "sort self test", __FILE__, __LINE__);
    } while (0);
    ka.release(); kb.release(); va.release(); vb.release();
    return rc;
}

} // extern "C"
