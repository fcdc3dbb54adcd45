// slab_selftest -- slab mode from C++ over NCCL (slab_host.h) against ONE handle processing the whole cloud: a synthetic room scan
// is cut into `gpus` contiguous shares (as if every GPU had recorded some of the scan positions), SlabRun segments it, and every
// rank's voxel labels / distances, merge log and labelled cloud must equal the single handle's bit for bit.
// usage: slab_selftest [--gpus N] [--points P] [--voxel v] [--seed s] [--threshold t] [--device-shares 0|1]
// (--device-shares 1: every rank's share is uploaded to its GPU first, as if the scans were already in HBM; the timed run starts from there)
// prints one JSON line (stage ms = max over ranks); exit code 0 = identical.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <string>
#include <vector>

#include "slab_host.h"

namespace {
struct Pt { float x, y, z, pad0; uint32_t bgra; uint32_t pad1[3]; };      // pcl::PointXYZRGBA, 32 bytes
static_assert(sizeof(Pt) == 32, "PointXYZRGBA layout");

struct Rng { uint64_t s; explicit Rng(uint64_t seed) : s(seed * 0x9E3779B97F4A7C15ull + 1) {}
    uint32_t next() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return (uint32_t)(s >> 32); }
    float uni() { return (float)(next() >> 8) * (1.0f / 16777216.0f); } };

// a room seen from a few scan positions: floor, back wall, side wall, boxes on the floor; colours per surface with noise
std::vector<Pt> make_room(int64_t n, uint64_t seed) {
    std::vector<Pt> pts((size_t)n);
    Rng rng(seed);
    for (int64_t i = 0; i < n; ++i) {
        Pt p; memset(&p, 0, sizeof p);
        const uint32_t which = rng.next() % 100;
        float x, y, z; uint32_t r, g, b;
        if (which < 40) { x = rng.uni() * 4 - 2; z = 1 + rng.uni() * 3; y = 1.0f + 0.002f * rng.uni(); r = 150; g = 120; b = 90; }            // floor
        else if (which < 65) { x = rng.uni() * 4 - 2; y = rng.uni() * 2 - 1; z = 4.0f + 0.002f * rng.uni(); r = 200; g = 200; b = 190; }      // back wall
        else if (which < 80) { x = -2.0f + 0.002f * rng.uni(); y = rng.uni() * 2 - 1; z = 1 + rng.uni() * 3; r = 90; g = 130; b = 170; }      // side wall
        else {                                                                                                                            // boxes
            const int k = (int)(which % 4);
            const float cx = -1.2f + 0.8f * (float)k, cz = 2.0f + 0.4f * (float)k, h = 0.3f + 0.1f * (float)k;
            const uint32_t face = rng.next() % 3;
            if (face == 0) { x = cx + rng.uni() * 0.4f; z = cz + rng.uni() * 0.4f; y = 1.0f - h; }
            else if (face == 1) { x = cx + rng.uni() * 0.4f; y = 1.0f - h * rng.uni(); z = cz; }
            else { x = cx; y = 1.0f - h * rng.uni(); z = cz + rng.uni() * 0.4f; }
            r = 60 + 50 * (uint32_t)k; g = 200 - 40 * (uint32_t)k; b = 40 + 30 * face;
        }
        if ((rng.next() & 1023u) == 0) x = std::numeric_limits<float>::quiet_NaN();                    // sensor drop-outs
        if ((rng.next() & 2047u) == 0) z = -z;                                                         // main(): z < 0 -> |z|
        const uint32_t nr = std::min(255u, r + rng.next() % 6), ng = std::min(255u, g + rng.next() % 6), nb = std::min(255u, b + rng.next() % 6);
        p.x = x; p.y = y; p.z = z; p.bgra = 0xff000000u | (nr << 16) | (ng << 8) | nb;
        pts[(size_t)i] = p;
    }
    return pts;
}

struct Result { std::vector<uint32_t> label; std::vector<float> dist; std::vector<uint32_t> mab; std::vector<float> mw; std::vector<uint32_t> mleft;
                std::vector<float> oxyz; std::vector<uint32_t> olab, ovox; f3ps_counts c; };
bool pull(f3ps_ctx* h, Result& r) {
    if (f3ps_get_counts(h, &r.c)) return false;
    const size_t V = (size_t)r.c.n_voxels, M = (size_t)r.c.n_merges, L = (size_t)r.c.n_labeled;
    r.label.resize(V); r.dist.resize(V); r.mab.resize(2 * M); r.mw.resize(M); r.mleft.resize(2 * M); r.oxyz.resize(3 * L); r.olab.resize(L); r.ovox.resize(L);
    if (V && f3ps_get_voxel_labels(h, r.label.data(), r.dist.data(), (int64_t)V)) return false;
    if (M && f3ps_get_merge_log(h, r.mab.data(), r.mw.data(), r.mleft.data(), (int64_t)M)) return false;
    if (L && f3ps_get_labeled_cloud(h, r.oxyz.data(), r.olab.data(), r.ovox.data(), (int64_t)L)) return false;
    return true;
}
template <typename T> bool same(const std::vector<T>& a, const std::vector<T>& b) { return a.size() == b.size() && (a.empty() || !memcmp(a.data(), b.data(), a.size() * sizeof(T))); }
}  // namespace

int main(int argc, char** argv) {
    int gpus = 0, device_shares = 0; int64_t n = 2000000; uint64_t seed = 7;
    f3ps_host::SlabParams p; p.voxel_res = 0.01f; p.seed_res = 0.1f; p.geometric_distance = 1; p.merging = 1;      // BASELINE config 5: -v 0.01 -s 0.1 --CVX --AL
    for (int i = 1; i + 1 < argc; i += 2) {
        const std::string k = argv[i];
        if (k == "--gpus") gpus = atoi(argv[i + 1]); else if (k == "--points") n = atoll(argv[i + 1]);
        else if (k == "--voxel") p.voxel_res = (float)atof(argv[i + 1]);
        else if (k == "--seed-res") p.seed_res = (float)atof(argv[i + 1]); else if (k == "--seed") seed = (uint64_t)atoll(argv[i + 1]);
        else if (k == "--threshold") p.threshold = (float)atof(argv[i + 1]);
        else if (k == "--device-shares") device_shares = atoi(argv[i + 1]);
        else { fprintf(stderr, "unknown option %s\n", k.c_str()); return 2; }
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) { fprintf(stderr, "slab_selftest: no CUDA device\n"); return 2; }
    if (gpus <= 0 || gpus > ndev) gpus = ndev;
    const std::vector<Pt> pts = make_room(n, seed);
    std::vector<int> devs; for (int d = 0; d < gpus; ++d) devs.push_back(d);
    f3ps_host::SlabRun run(devs);
    if (!run.ok()) { fprintf(stderr, "slab_selftest: %s\n", run.init_error().c_str()); return 2; }
    std::vector<f3ps_host::SlabShare> shares((size_t)gpus);
    for (int r = 0; r < gpus; ++r) {                       // uneven contiguous shares
        const int64_t lo = n * r / gpus + (r ? n / (7 * gpus) : 0), hi = r + 1 < gpus ? n * (r + 1) / gpus + n / (7 * gpus) : n;
        shares[(size_t)r].points = pts.data() + lo; shares[(size_t)r].n = hi - lo; shares[(size_t)r].stride = 32;
        if (device_shares && hi > lo) {
            void* d = nullptr;
            if (cudaSetDevice(r) != cudaSuccess || cudaMalloc(&d, (size_t)(hi - lo) * 32) != cudaSuccess ||
                cudaMemcpy(d, pts.data() + lo, (size_t)(hi - lo) * 32, cudaMemcpyHostToDevice) != cudaSuccess) { fprintf(stderr, "slab_selftest: upload of share %d failed\n", r); return 2; }
            shares[(size_t)r].points = d; shares[(size_t)r].on_device = true;
        }
    }
    int rc = 0;
    for (int rep = 0; rep < 2 && !rc; ++rep) rc = run.run(shares, p);     // twice: the second run is the timed one (buffers allocated, NCCL warm)
    if (rc) { for (int r = 0; r < gpus; ++r) if (!run.info(r).error.empty()) fprintf(stderr, "rank %d: %s\n", r, run.info(r).error.c_str()); return 1; }
    // one handle, the whole cloud
    f3ps_ctx* one = nullptr;
    cudaSetDevice(0);
    if (f3ps_create(0, nullptr, &one)) { fprintf(stderr, "f3ps_create failed\n"); return 2; }
    f3ps_set_vccs_params(one, p.voxel_res, p.seed_res, p.color_imp, p.spatial_imp, p.normal_imp, p.use_transform, p.fold_negative_z);
    f3ps_set_merge_params(one, p.color_distance, p.geometric_distance, p.merging, p.lambda, p.bins);
    if (f3ps_set_input(one, pts.data(), n, 32, 0) || f3ps_run(one, p.threshold) || f3ps_sync(one)) { fprintf(stderr, "single handle: %s\n", f3ps_last_error(one)); return 1; }
    Result ref; if (!pull(one, ref)) { fprintf(stderr, "single handle: read-back failed\n"); return 1; }
    float one_total = 0; f3ps_stage_ms(one, F3PS_STAGE_TOTAL, &one_total);
    bool identical = true; std::string diff;
    for (int r = 0; r < gpus; ++r) {
        Result got; if (!pull(run.handle(r), got)) { identical = false; diff += " rank" + std::to_string(r) + ":readback"; continue; }
        const bool ok = same(got.label, ref.label) && same(got.dist, ref.dist) && same(got.mab, ref.mab) && same(got.mw, ref.mw) && same(got.mleft, ref.mleft) &&
                        same(got.oxyz, ref.oxyz) && same(got.olab, ref.olab) && same(got.ovox, ref.ovox) && got.c.n_supervoxels == ref.c.n_supervoxels && got.c.n_edges == ref.c.n_edges;
        if (!ok) { identical = false; diff += " rank" + std::to_string(r); }
    }
    std::map<std::string, float> ms; std::vector<std::string> order; uint64_t bytes = 0;
    for (int r = 0; r < gpus; ++r) {
        for (auto& kv : run.info(r).stage_ms) { if (!ms.count(kv.first)) order.push_back(kv.first); ms[kv.first] = std::max(ms[kv.first], kv.second); }
        bytes = std::max(bytes, run.info(r).bytes_exchanged);
    }
    printf("{\"tool\": \"slab_selftest\", \"host\": \"c++/nccl\", \"gpus\": %d, \"points\": %lld, \"V\": %lld, \"S\": %d, \"E\": %d, \"merges\": %d, \"sweeps\": %d, "
           "\"device_shares\": %s, \"identical_to_one_handle\": %s, \"bytes_exchanged_max_rank\": %llu, \"one_handle_total_ms\": %.3f, \"stage_ms\": {",
           gpus, (long long)n, (long long)run.info(0).V, ref.c.n_supervoxels, ref.c.n_edges, ref.c.n_merges, run.info(0).sweeps,
           device_shares ? "true" : "false", identical ? "true" : "false", (unsigned long long)bytes, one_total);
    for (size_t i = 0; i < order.size(); ++i) printf("%s\"%s\": %.3f", i ? ", " : "", order[i].c_str(), ms[order[i]]);
    printf("}}\n");
    if (!identical) fprintf(stderr, "slab_selftest: differs from the single handle on:%s\n", diff.c_str());
    f3ps_destroy(one);
    return identical ? 0 : 1;
}
