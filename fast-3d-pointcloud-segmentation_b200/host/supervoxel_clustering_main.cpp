// supervoxel_clustering -- the reference's CLI (src/supervoxel_clustering.cpp:136-476) over the f3ps CUDA path.
// Same flags, same defaults, same quirks for the hot path:
//   {-d <dir> | -p <file>}  -v -s -c -z -n  -t  --RGB --CVX --ML [l] --AL --EQ [bins]  --NT --V
// Without -t the threshold sweep of the reference runs (41 thresholds against the ground truth, best F-score, :428-438).
// -r <label> drops the points of one ground-truth label (:295-298, 329-333), -f <name> names the seven score files
// <name>_{voi,precision,recall,fscore,wov,fpr,fnr}.csv (:194-196, 478-518); the final scores are printed as :520-557 does.
// Not built: the interactive viewer.
// Additions: --no-eval skips the evaluation of the final segmentation, -o <file.pcd> writes the labelled voxel cloud (per
// file "<stem>_<o>" in a -d sweep), --facade routes through the Clustering / SupervoxelClustering
// classes instead of the fused path, --gpus N shards the files of a -d sweep over N GPUs (no collective), --inflight K =
// files per group of a sweep: K1..K6 of a file on its own handle + stream, ONE merge launch per group (f3ps_merge_batch),
// the next group's front stages overlapping it.  --levels t1,t2,... prints the segmentation at several thresholds from one
// extra merge replay, --point-labels <file.pcd> writes the input cloud with every point's segment (one file per level),
// --segments <file.csv> writes one row per segment (point and voxel counts, bounds, centroid, mean colour) of every level.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <fstream>
#include <map>
#include <mutex>
#include <memory>
#include <thread>

#include "pcd_io.h"
#include "slab_host.h"
#include "supervoxel_clustering/clustering.h"

namespace {
// pcl::console::find_switch / parse_argument semantics: exact strcmp match, value = the next argv
bool find_switch(int argc, char** argv, const char* name) {
    for (int i = 1; i < argc; ++i) if (strcmp(argv[i], name) == 0) return true;
    return false;
}
int find_argument(int argc, char** argv, const char* name) {
    for (int i = 1; i < argc; ++i) if (strcmp(argv[i], name) == 0) return i;
    return -1;
}
bool parse(int argc, char** argv, const char* name, float& v) { int i = find_argument(argc, argv, name); if (i > 0 && i + 1 < argc) { v = (float)atof(argv[i + 1]); return true; } return false; }
bool parse(int argc, char** argv, const char* name, int& v) { int i = find_argument(argc, argv, name); if (i > 0 && i + 1 < argc) { v = atoi(argv[i + 1]); return true; } return false; }
bool parse(int argc, char** argv, const char* name, std::string& v) { int i = find_argument(argc, argv, name); if (i > 0 && i + 1 < argc) { v = argv[i + 1]; return true; } return false; }

struct Options {
    float voxel_resolution = 0.008f, seed_resolution = 0.08f, color_importance = 0.2f, spatial_importance = 0.4f, normal_importance = 1.0f;
    float thresh = 0; bool thresh_specified = true; bool rgb = false, cvx = false, ml = false, al = false, eq = false, disable_transform = false, verbose = false, facade = false;
    float lambda = 0; int bin_num = 0; std::string out;
    bool remove_label = false; uint32_t label_to_be_removed = 0; std::string test_filename = "test"; bool eval = true;
    std::vector<float> levels; std::string point_labels, segments;
};
struct FileScores { bool have_best = false; f3ps_performance best; std::vector<std::pair<float, f3ps_performance>> all; };

void usage(const char* a0) {
    printf("Syntax is: %s {-d <direcory-of-pcd-files> OR -p <pcd-file>} [arguments] \n\n"
           "\tSUPERVOXEL optional arguments: \n"
           "\t -v <voxel-resolution>          (default: 0.008) \n\t -s <seed-resolution>           (default: 0.08) \n"
           "\t -c <color-weight>              (default: 0.2) \n\t -z <spatial-weight>            (default: 0.4) \n"
           "\t -n <normal-weight>             (default: 1.0) \n\n"
           "\tSEGMENTATION optional arguments: \n"
           "\t -t <threshold>                 (default: auto)\n"
           "\t --RGB                          (RGB colour distance instead of L*A*B* CIEDE2000) \n"
           "\t --CVX                          (convexity criterion on the geometric distance) \n"
           "\t --ML [manual-lambda] *         (Manual Lambda; lambda=0.5 when no value is given) \n"
           "\t --AL                 *         (Adaptive Lambda, the default) \n"
           "\t --EQ [bins-number]   *         (Equalization; 500 bins when no value is given -- the reference's text says 200) \n"
           "\t  * only one of these can be passed at a time \n\n"
           "\tOTHER optional arguments: \n"
           "\t -r <label-to-be-removed>       (if ground-truth is provided, removes all points with the given label from the ground-truth)\n"
           "\t -f <test-results-filename>     (name of the test results files; 'test' if not given)\n"
           "\t --no-eval                      (skips the evaluation of the final segmentation)\n"
           "\t --NT                           (disables the single camera transform) \n"
           "\t --V                            (verbose: prints the merge sequence) \n"
           "\t -o <file.pcd>                  (writes the labelled voxel cloud) \n"
           "\t --levels <t1,t2,...>           (prints the segment counts at these ascending thresholds, one extra merge replay) \n"
           "\t --point-labels <file.pcd>      (writes every input point with its segment; with --levels one file <stem>_<k>.pcd per level)\n"
           "\t --segments <file.csv>          (writes one row per segment: counts, bounds, centroid and mean colour of its points; with\n"
           "\t                                 --levels the segments of every level in the one file) \n"
           "\t --facade                       (runs through the Clustering / SupervoxelClustering classes) \n"
           "\t --gpus <N>                     (shards the files of -d over N GPUs) \n"
           "\t --inflight <K>                 (frames in flight per GPU during a -d sweep, default 8) \n"
           "\t --slabs <N>                    (with -p and -t: ONE cloud cut into N spatial slabs, one per GPU, exchanges over NCCL;\n"
           "\t                                 same result as one GPU; no evaluation against ground truth in this mode) \n", a0);
}

// main()'s input clean-up (src/supervoxel_clustering.cpp:315-337): z<0 -> |z|; with -r, the points of that label and the points
// with a NaN z are dropped (has_label is hard-coded true there, so the test reduces to this)
void clean_input(pcl::PointCloud<pcl::PointXYZRGBL>& input, const Options& o) {
    for (auto& p : input.points) if (p.z < 0) p.z = std::abs(p.z);
    if (!o.remove_label) return;
    pcl::PointCloud<pcl::PointXYZRGBL> kept;
    for (auto& p : input.points) if (p.label != o.label_to_be_removed && !std::isnan(p.z)) kept.push_back(p);
    input = kept;
}

// Testing(segmentation.get_labeled_cloud(), truth_cloud).eval_performance() (:456-457) for the handle's current segmentation:
// the labelled voxel cloud against the ground-truth voxel labels, contingency table on the device
f3ps_performance final_scores(f3ps::Handle& h, const std::vector<uint32_t>& truth, int n_labeled, const std::vector<uint32_t>& lab, const std::vector<uint32_t>& vox) {
    std::map<uint32_t, uint32_t> dense;
    for (uint32_t t : truth) dense[t] = 0;
    uint32_t nt = 0; for (auto& kv : dense) kv.second = nt++;
    std::vector<uint64_t> tsizes(nt, 0);
    for (uint32_t t : truth) tsizes[dense[t]]++;
    uint32_t ns = 0; for (int i = 0; i < n_labeled; ++i) ns = std::max(ns, lab[(size_t)i] + 1);
    std::vector<uint32_t> tl((size_t)n_labeled);
    for (int i = 0; i < n_labeled; ++i) tl[(size_t)i] = dense[truth[vox[(size_t)i]]];
    f3ps_performance pf{0, 0, 0, 0, 0, 0, 0};
    if (n_labeled > 0 && !truth.empty())
        h.check(f3ps_eval_label_pairs(h.get(), lab.data(), tl.data(), n_labeled, (int32_t)ns, (int32_t)nt, tsizes.data(), (int64_t)truth.size(), &pf));
    return pf;
}

// manageAllPerformances (:478-518): seven files, one line per input file, one ';'-terminated value per threshold
void manage_all_performances(const std::vector<FileScores>& scores, const std::string& filename) {
    const char* names[7] = {"voi", "precision", "recall", "fscore", "wov", "fpr", "fnr"};
    for (int k = 0; k < 7; ++k) {
        std::ofstream f((filename + "_" + names[k] + ".csv").c_str());
        for (const FileScores& s : scores) {
            if (s.all.empty()) continue;                                 // a file clustered with -t has no sweep (all_performances gets no entry, :428-431)
            for (auto& kv : s.all) {
                const f3ps_performance& p = kv.second;
                const float v[7] = {p.voi, p.precision, p.recall, p.fscore, p.wov, p.fpr, p.fnr};
                f << v[k] << ";";
            }
            f << "\n";
        }
    }
}
// printBestPerformances (:520-557).  The reference's average uses an integer 1/count, so only the first file counts
// (SURVEY.md D.7, a reporting bug); the running mean below is the intended one.
void print_best_performances(const std::vector<FileScores>& scores) {
    std::vector<f3ps_performance> best;
    for (const FileScores& s : scores) if (s.have_best) best.push_back(s.best);
    if (best.empty()) return;
    if (best.size() == 1) {
        const f3ps_performance& p = best.back();
        printf("Scores:\nVOI\t%f\nPrec.\t%f\nRecall\t%f\nF-score\t%f\nWOv\t%f\nFPR\t%f\nFNR\t%f\n", p.voi, p.precision, p.recall, p.fscore, p.wov, p.fpr, p.fnr);
        return;
    }
    float m[7] = {0, 0, 0, 0, 0, 0, 0}; int count = 0;
    for (const f3ps_performance& p : best) {
        ++count;
        const float v[7] = {p.voi, p.precision, p.recall, p.fscore, p.wov, p.fpr, p.fnr};
        for (int k = 0; k < 7; ++k) m[k] = m[k] + (1.0f / count) * (v[k] - m[k]);
    }
    printf("Average scores:\nVOI\t%f\nPrec.\t%f\nRecall\t%f\nF-score\t%f\nWOv\t%f\nFPR\t%f\nFNR\t%f\n", m[0], m[1], m[2], m[3], m[4], m[5], m[6]);
}

// Ground-truth voxelisation (src/supervoxel_clustering.cpp:387-400): the reference colours the truth cloud with the Glasbey
// table, runs VCCS on it and maps the voxel colours back to labels (color2label: labels by first occurrence in voxel order,
// src/clustering.cpp:823-846).  A voxel whose points share one label keeps that label's colour; a mixed voxel gets the mean
// colour, i.e. a class of its own shared with the voxels of the same label mixture.  PCL's Glasbey table is not in the
// reference tree, so mixtures are keyed by their label proportions instead of the blended colour (equal unless two
// different mixtures happen to blend to the same 8-bit colour).
std::vector<uint32_t> voxelise_truth(const std::vector<int32_t>& point_voxel, const pcl::PointCloud<pcl::PointXYZRGBL>& input, size_t V) {
    std::vector<std::map<uint32_t, uint32_t>> mix(V);
    for (size_t i = 0; i < point_voxel.size(); ++i) if (point_voxel[i] >= 0) mix[(size_t)point_voxel[i]][input.points[i].label]++;
    std::map<std::vector<std::pair<uint32_t, uint32_t>>, uint32_t> classes;      // color2label's std::map<float, uint32_t>
    std::vector<uint32_t> truth(V, 0);
    for (size_t v = 0; v < V; ++v) {
        std::vector<std::pair<uint32_t, uint32_t>> key(mix[v].begin(), mix[v].end());
        uint32_t g = 0;
        for (auto& kv : key) { uint32_t a = kv.second, b = g; while (b) { uint32_t t = a % b; a = b; b = t; } g = a; }
        if (key.size() == 1) key[0].second = 1; else for (auto& kv : key) kv.second /= std::max(1u, g);
        auto it = classes.find(key);
        if (it == classes.end()) it = classes.insert(std::make_pair(key, (uint32_t)classes.size())).first;
        truth[v] = it->second;
    }
    return truth;
}

// Clustering::all_thresh + best_thresh (src/clustering.cpp:691-774) as main() uses them (:428-438): one merge replay on the device
float auto_threshold(f3ps::Handle& h, const std::vector<uint32_t>& truth, std::string& report, FileScores* fs) {
    const float start_thresh = 0.8f, end_thresh = 1.0f, step_thresh = 0.005f;   // globals of the reference (:76-78)
    std::vector<float> thr(1, start_thresh);
    for (float t = start_thresh + step_thresh; t <= end_thresh; t += step_thresh) thr.push_back(t);
    std::vector<f3ps_performance> perf(thr.size());
    h.check(f3ps_eval_thresholds(h.get(), truth.data(), (int64_t)truth.size(), nullptr, 0, thr.data(), (int)thr.size(), perf.data(), nullptr, nullptr));
    char buf[256];
    snprintf(buf, sizeof buf, "Testing thresholds from %f to %f (step %f)\n", start_thresh, end_thresh, step_thresh); report += buf;
    float best_t = 0; f3ps_performance best{0, 0, 0, 0, 0, 0, 0};
    for (size_t k = 0; k < thr.size(); ++k) {
        snprintf(buf, sizeof buf, "<T, Fscore, voi, wov> = <%f, %f, %f, %f>\n", thr[k], perf[k].fscore, perf[k].voi, perf[k].wov); report += buf;
        if (perf[k].fscore > best.fscore) { best = perf[k]; best_t = thr[k]; }
        if (fs) fs->all.push_back(std::make_pair(thr[k], perf[k]));
    }
    snprintf(buf, sizeof buf, "Using best threshold: %f (F-score %f, voi %f)\n", best_t, best.fscore, best.voi); report += buf;
    return best_t;
}

// ---- a -d sweep with -t: front stages per file, one merge launch per group ---------------------------------------
struct SweepJob {
    std::string file; pcl::PointCloud<pcl::PointXYZRGBA>::Ptr cloud; std::chrono::steady_clock::time_point t0;
    pcl::PointCloud<pcl::PointXYZRGBL> input;                            // kept for the ground-truth labels of the evaluation
};
void sweep_front(SweepJob& j, const Options& o, f3ps::Handle& h) {
    pcl::PointCloud<pcl::PointXYZRGBL>& input = j.input;
    f3ps::loadPCDFile(j.file, input);                                    // return value ignored, as in the reference (:313)
    j.cloud.reset(new pcl::PointCloud<pcl::PointXYZRGBA>());
    clean_input(input, o);                                               // :315-337
    pcl::copyPointCloud(input, *j.cloud);
    const int merging = o.ml ? F3PS_MANUAL_LAMBDA : (o.eq ? F3PS_EQUALIZATION : F3PS_ADAPTIVE_LAMBDA);
    const float lam = (o.ml && o.lambda != 0) ? o.lambda : 0.5f;
    const int bins = (o.eq && o.bin_num != 0) ? o.bin_num : 500;
    j.t0 = std::chrono::steady_clock::now();
    h.check(f3ps_set_vccs_params(h.get(), o.voxel_resolution, o.seed_resolution, o.color_importance, o.spatial_importance,
                                 o.normal_importance, o.disable_transform ? 0 : 1, 0));
    h.check(f3ps_set_merge_params(h.get(), o.rgb ? F3PS_RGB_EUCL : F3PS_LAB_CIEDE00, o.cvx ? F3PS_CONVEX_NORMALS_DIFF : F3PS_NORMALS_DIFF, merging, lam, bins));
    h.check(f3ps_set_input(h.get(), j.cloud->points.data(), (int64_t)j.cloud->size(), 32, 0));
    h.check(f3ps_extract(h.get()));
    h.check(f3ps_graph(h.get()));
}
void sweep_back(SweepJob& j, const Options& o, f3ps::Handle& h, int device, std::string& report, FileScores& fs) {
    f3ps_counts n; h.check(f3ps_get_counts(h.get(), &n));
    if (o.eval && n.n_labeled > 0) {
        std::vector<int32_t> pv((size_t)n.n_points);
        h.check(f3ps_get_point_voxel(h.get(), pv.data(), n.n_points));
        std::vector<float> xyz(3 * (size_t)n.n_labeled); std::vector<uint32_t> lab(n.n_labeled), vox(n.n_labeled);
        h.check(f3ps_get_labeled_cloud(h.get(), xyz.data(), lab.data(), vox.data(), n.n_labeled));
        fs.best = final_scores(h, voxelise_truth(pv, j.input, (size_t)n.n_voxels), n.n_labeled, lab, vox); fs.have_best = true;
    }
    float stage[9] = {0};
    for (int s = 0; s < 9; ++s) f3ps_stage_ms(h.get(), s, &stage[s]);
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - j.t0).count();
    char buf[512];
    snprintf(buf, sizeof buf, "Loading pointcloud from PCD file '%s'...\nFound %d supervoxels\n", j.file.c_str(), n.n_supervoxels); report += buf;
    if (o.verbose) {
        std::vector<uint32_t> ab(2 * (size_t)n.n_merges), left(2 * (size_t)n.n_merges); std::vector<float> w(n.n_merges);
        h.check(f3ps_get_merge_log(h.get(), ab.data(), w.data(), left.data(), (int64_t)n.n_merges));
        for (int m = 0; m < n.n_merges; ++m) { snprintf(buf, sizeof buf, "left: %de/%dp - w: %f - [%d, %d]...OK\n", left[2 * m], left[2 * m + 1], w[m], ab[2 * m], ab[2 * m + 1]); report += buf; }
    }
    snprintf(buf, sizeof buf, "Clustering complete: %zu points -> %d merges -> %d segments over %d voxels in %.3f ms (GPU %d)\n",
             j.cloud->size(), n.n_merges, n.n_segments, n.n_labeled, ms, device); report += buf;
    snprintf(buf, sizeof buf, "  stage ms: voxelize %.3f neighbors %.3f normals %.3f seeds %.3f expand %.3f graph %.3f merge %.3f total %.3f\n",
             stage[0], stage[1], stage[2], stage[3], stage[4], stage[5], stage[6], stage[7]); report += buf;
    j.cloud.reset(); j.input.clear();
}
// one GPU's share of the files: groups of `group` files, two handle sets alternate
void sweep_device(const std::vector<size_t>& mine, const std::vector<std::string>& files, const Options& o, int device, int group,
                  std::vector<std::string>& reports, std::vector<FileScores>& scores, std::string& first_error, std::mutex& emu) {
    auto fail = [&](const std::exception& e) { std::lock_guard<std::mutex> g(emu); if (first_error.empty()) first_error = e.what(); };
    try {
        const int threads = (int)std::max(2u, std::min<unsigned>((unsigned)group, std::thread::hardware_concurrency()));
        std::vector<std::unique_ptr<f3ps::Handle>> sets[2];
        for (int s = 0; s < 2; ++s) for (int k = 0; k < group; ++k) {
            sets[s].emplace_back(new f3ps::Handle(device));
            f3ps_set_blocking_wait(sets[s].back()->get(), 1);
            f3ps_set_expand_kernel(sets[s].back()->get(), 2, 8);          // sweeps: K5 of a file as one cluster of 8 CTAs, the files side by side
        }
        std::vector<SweepJob> jobs[2];
        std::thread back;
        for (size_t g0 = 0, gi = 0; g0 < mine.size(); g0 += (size_t)group, ++gi) {
            const size_t g1 = std::min(mine.size(), g0 + (size_t)group);
            const int si = (int)(gi & 1);
            // the set this group is about to use was merged two groups ago; the previous group's merge is still running
            jobs[si].assign(g1 - g0, SweepJob());
            for (size_t k = g0; k < g1; ++k) jobs[si][k - g0].file = files[mine[k]];
            std::vector<std::thread> th;
            for (int w = 0; w < threads; ++w) th.emplace_back([&, w]() {
                try { for (size_t k = (size_t)w; k < g1 - g0; k += (size_t)threads) sweep_front(jobs[si][k], o, *sets[si][k]); }
                catch (const std::exception& e) { fail(e); }
            });
            for (auto& t : th) t.join();
            if (back.joinable()) back.join();
            { std::lock_guard<std::mutex> g(emu); if (!first_error.empty()) return; }
            back = std::thread([&, si, g0, g1]() {
                try {
                    std::vector<f3ps_ctx*> ctxs;
                    for (size_t k = 0; k < g1 - g0; ++k) ctxs.push_back(sets[si][k]->get());
                    sets[si][0]->check(f3ps_merge_batch(ctxs.data(), (int)ctxs.size(), o.thresh));   // Clustering::cluster of every file of the group (:443)
                    for (size_t k = 0; k < g1 - g0; ++k) sweep_back(jobs[si][k], o, *sets[si][k], device, reports[mine[g0 + k]], scores[mine[g0 + k]]);
                } catch (const std::exception& e) { fail(e); }
            });
        }
        if (back.joinable()) back.join();
    } catch (const std::exception& e) { fail(e); }
}

int process_file(const std::string& file, const Options& o, int device, std::string& report, f3ps::Handle* worker, FileScores& fs, bool in_sweep) {
    pcl::PointCloud<pcl::PointXYZRGBL> input;
    f3ps::loadPCDFile(file, input);                                      // return value ignored, as in the reference (:313)
    pcl::PointCloud<pcl::PointXYZRGBA>::Ptr cloud(new pcl::PointCloud<pcl::PointXYZRGBA>());
    clean_input(input, o);                                               // :315-337
    pcl::copyPointCloud(input, *cloud);
    const int merging = o.ml ? F3PS_MANUAL_LAMBDA : (o.eq ? F3PS_EQUALIZATION : F3PS_ADAPTIVE_LAMBDA);
    const float lam = (o.ml && o.lambda != 0) ? o.lambda : 0.5f;         // --ML 0 means "unset" (:417)
    const int bins = (o.eq && o.bin_num != 0) ? o.bin_num : 500;         // --EQ 0 means "unset" (:421)
    auto t0 = std::chrono::steady_clock::now();
    pcl::PointCloud<pcl::PointXYZL>::Ptr labeled(new pcl::PointCloud<pcl::PointXYZL>());
    size_t n_sv = 0, n_seg = 0, n_merges = 0; float stage[9] = {0};
    float thresh = o.thresh;                                                 // of the final segmentation: -t or the sweep's choice
    std::vector<MergeStep> log;
    std::unique_ptr<f3ps::Handle> local;                                     // -p: a handle of its own; sweeps reuse the worker's (buffers stay allocated)
    f3ps::Handle* hp = nullptr;
    if (o.facade) {
        pcl::SupervoxelClustering<pcl::PointXYZRGBA> super(o.voxel_resolution, o.seed_resolution, device);
        super.setUseSingleCameraTransform(!o.disable_transform);
        super.setInputCloud(cloud);
        super.setColorImportance(o.color_importance); super.setSpatialImportance(o.spatial_importance); super.setNormalImportance(o.normal_importance);
        std::map<uint32_t, pcl::Supervoxel<pcl::PointXYZRGBA>::Ptr> supervoxel_clusters;
        super.extract(supervoxel_clusters);
        std::multimap<uint32_t, uint32_t> label_adjacency;
        super.getSupervoxelAdjacency(label_adjacency);
        Clustering segmentation;
        if (o.rgb) segmentation.set_delta_c(RGB_EUCL);
        if (o.cvx) segmentation.set_delta_g(CONVEX_NORMALS_DIFF);
        if (o.ml) { segmentation.set_merging(MANUAL_LAMBDA); if (o.lambda != 0) segmentation.set_lambda(o.lambda); }
        else if (o.eq) { segmentation.set_merging(EQUALIZATION); if (o.bin_num != 0) segmentation.set_bins_num((short)o.bin_num); }
        segmentation.set_initialstate(supervoxel_clusters, label_adjacency);
        segmentation.cluster(o.thresh);
        labeled = segmentation.get_labeled_cloud();
        if (o.eval && !labeled->empty()) {                                  // the reference's own sequence (:386-400, 456-457) through the classes
            pcl::PointCloud<pcl::PointXYZL>::Ptr truth_cloud(new pcl::PointCloud<pcl::PointXYZL>());
            pcl::copyPointCloud(input, *truth_cloud);
            pcl::PointCloud<pcl::PointXYZRGBA>::Ptr colored_truth_cloud = Clustering::label2color(truth_cloud);
            pcl::SupervoxelClustering<pcl::PointXYZRGBA> super_label(o.voxel_resolution, o.seed_resolution, device);
            super_label.setUseSingleCameraTransform(!o.disable_transform);
            super_label.setInputCloud(colored_truth_cloud);
            super_label.setColorImportance(o.color_importance); super_label.setSpatialImportance(o.spatial_importance); super_label.setNormalImportance(o.normal_importance);
            std::map<uint32_t, pcl::Supervoxel<pcl::PointXYZRGBA>::Ptr> supervoxel_label_clusters;
            super_label.extract(supervoxel_label_clusters);
            truth_cloud = Clustering::color2label(super_label.getVoxelCentroidCloud());
            Testing test(labeled, truth_cloud);
            const performanceSet ps = test.eval_performance();
            fs.best = f3ps_performance{ps.voi, ps.precision, ps.recall, ps.fscore, ps.wov, ps.fpr, ps.fnr}; fs.have_best = true;
        }
        n_sv = supervoxel_clusters.size(); n_seg = segmentation.get_currentstate().first.size();
        log = segmentation.get_merge_log(); n_merges = log.size();
    } else {
        if (!worker) local.reset(new f3ps::Handle(device));
        hp = worker ? worker : local.get();
        f3ps::Handle& h = *hp;
        h.check(f3ps_set_vccs_params(h.get(), o.voxel_resolution, o.seed_resolution, o.color_importance, o.spatial_importance,
                                     o.normal_importance, o.disable_transform ? 0 : 1, 0));
        h.check(f3ps_set_merge_params(h.get(), o.rgb ? F3PS_RGB_EUCL : F3PS_LAB_CIEDE00, o.cvx ? F3PS_CONVEX_NORMALS_DIFF : F3PS_NORMALS_DIFF, merging, lam, bins));
        h.check(f3ps_set_input(h.get(), cloud->points.data(), (int64_t)cloud->size(), 32, 0));
        std::vector<uint32_t> truth;
        if (o.thresh_specified && !o.eval) h.check(f3ps_run(h.get(), thresh));
        else {
            h.check(f3ps_extract(h.get())); h.check(f3ps_graph(h.get()));
            f3ps_counts n0; h.check(f3ps_get_counts(h.get(), &n0));
            std::vector<int32_t> pv((size_t)n0.n_points);
            h.check(f3ps_get_point_voxel(h.get(), pv.data(), n0.n_points));
            truth = voxelise_truth(pv, input, (size_t)n0.n_voxels);          // :386-400
            if (!o.thresh_specified) thresh = auto_threshold(h, truth, report, &fs);   // no -t: the reference's threshold sweep (:428-438)
            h.check(f3ps_merge(h.get(), thresh));                           // main() (re-)clusters at the chosen threshold (:443)
        }
        f3ps_counts n; h.check(f3ps_get_counts(h.get(), &n));
        n_sv = n.n_supervoxels; n_seg = n.n_segments; n_merges = n.n_merges;
        std::vector<float> xyz(3 * (size_t)n.n_labeled); std::vector<uint32_t> lab(n.n_labeled), vox(n.n_labeled);
        h.check(f3ps_get_labeled_cloud(h.get(), xyz.data(), lab.data(), vox.data(), n.n_labeled));
        labeled->resize(n.n_labeled);
        for (int i = 0; i < n.n_labeled; ++i) { auto& p = labeled->points[i]; p.x = xyz[3 * i]; p.y = xyz[3 * i + 1]; p.z = xyz[3 * i + 2]; p.label = lab[i]; }
        if (o.eval && n.n_labeled > 0) { fs.best = final_scores(h, truth, n.n_labeled, lab, vox); fs.have_best = true; }   // :456-457
        for (int s = 0; s < 9; ++s) f3ps_stage_ms(h.get(), s, &stage[s]);
        if (o.verbose) {
            std::vector<uint32_t> ab(2 * n_merges), left(2 * n_merges); std::vector<float> w(n_merges);
            h.check(f3ps_get_merge_log(h.get(), ab.data(), w.data(), left.data(), (int64_t)n_merges));
            for (size_t m = 0; m < n_merges; ++m) log.push_back(MergeStep{ab[2 * m], ab[2 * m + 1], w[m], left[2 * m], left[2 * m + 1]});
        }
    }
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    char buf[512];
    snprintf(buf, sizeof buf, "Loading pointcloud from PCD file '%s'...\nFound %zu supervoxels\n", file.c_str(), n_sv); report += buf;
    if (o.verbose) for (auto& m : log) { snprintf(buf, sizeof buf, "left: %de/%dp - w: %f - [%d, %d]...OK\n", m.edges_left, m.regions_left, m.w, m.a, m.b); report += buf; }
    snprintf(buf, sizeof buf, "Clustering complete: %zu points -> %zu merges -> %zu segments over %zu voxels in %.3f ms (GPU %d)\n",
             cloud->size(), n_merges, n_seg, labeled->size(), ms, device); report += buf;
    if (!o.facade) { snprintf(buf, sizeof buf, "  stage ms: voxelize %.3f neighbors %.3f normals %.3f seeds %.3f expand %.3f graph %.3f merge %.3f total %.3f\n",
                              stage[0], stage[1], stage[2], stage[3], stage[4], stage[5], stage[6], stage[7]); report += buf; }
    // a sweep writes one file per input: <stem>_<o> next to -o's path
    auto per_file = [&](const std::string& name) {
        if (!in_sweep) return name;
        const std::filesystem::path op(name);
        return (op.parent_path() / (std::filesystem::path(file).stem().string() + "_" + op.filename().string())).string();
    };
    if (!o.out.empty()) f3ps::savePCDFileASCII(per_file(o.out), *labeled);
    if (hp && (!o.levels.empty() || !o.point_labels.empty() || !o.segments.empty())) {         // one more replay; the segmentation above stays f3ps_merge(thresh)'s
        f3ps::Handle& h = *hp;
        const std::vector<float> thr = o.levels.empty() ? std::vector<float>(1, thresh) : o.levels;
        h.check(f3ps_merge_levels(h.get(), thr.data(), (int)thr.size()));
        const int L = (int)thr.size();
        std::vector<int32_t> nm(L), ns(L);
        h.check(f3ps_get_levels(h.get(), nullptr, nullptr, nm.data(), ns.data(), L));
        if (!o.levels.empty())
            for (int k = 0; k < L; ++k) { snprintf(buf, sizeof buf, "level %d: threshold %f -> %d merges -> %d segments\n", k, thr[k], nm[k], ns[k]); report += buf; }
        if (!o.point_labels.empty()) {
            const size_t N = cloud->size();
            std::vector<uint32_t> lab((size_t)L * N);
            h.check(f3ps_get_level_point_labels(h.get(), lab.data(), (int64_t)lab.size(), 0));
            const std::filesystem::path base(per_file(o.point_labels));
            pcl::PointCloud<pcl::PointXYZL> pc;
            pc.resize(N);
            for (int k = 0; k < L; ++k) {
                for (size_t i = 0; i < N; ++i) {
                    const auto& q = cloud->points[i]; auto& p = pc.points[i];
                    p.x = q.x; p.y = q.y; p.z = q.z; p.label = lab[(size_t)k * N + i];
                }
                const std::string name = o.levels.empty() ? base.string()
                    : (base.parent_path() / (base.stem().string() + "_" + std::to_string(k) + base.extension().string())).string();
                f3ps::savePCDFileASCII(name, pc);
            }
        }
        if (!o.segments.empty()) {
            const std::string name = per_file(o.segments);
            FILE* f = fopen(name.c_str(), "w");
            if (!f) throw std::runtime_error("cannot write " + name);
            fprintf(f, "level,threshold,segment,region_label,n_points,n_voxels,min_x,min_y,min_z,max_x,max_y,max_z,cx,cy,cz,r,g,b\n");
            for (int k = 0; k < L; ++k) {
                std::vector<f3ps_segment_info> info((size_t)ns[k]);
                h.check(f3ps_get_segment_info(h.get(), k, info.data(), ns[k]));
                for (int j = 0; j < ns[k]; ++j) {
                    const f3ps_segment_info& q = info[(size_t)j];
                    fprintf(f, "%d,%.9g,%d,%u,%lld,%d,%.9g,%.9g,%.9g,%.9g,%.9g,%.9g,%.9g,%.9g,%.9g,%.9g,%.9g,%.9g\n", k, thr[k], j, q.region_label,
                            (long long)q.n_points, q.n_voxels, q.min_xyz[0], q.min_xyz[1], q.min_xyz[2], q.max_xyz[0], q.max_xyz[1], q.max_xyz[2],
                            q.centroid[0], q.centroid[1], q.centroid[2], q.mean_rgb[0], q.mean_rgb[1], q.mean_rgb[2]);
                }
            }
            fclose(f);
        }
    }
    return 0;
}
} // namespace

// --slabs N: one very large cloud over N GPUs (BASELINE config 5).  The reference's call sequence for the file (:313-367, 408-449)
// with SupervoxelClustering::extract + Clustering::cluster replaced by f3ps_host::SlabRun (slab_host.h); rank 0's handle reports.
int run_slabs(const std::string& file, const Options& o, int slabs) {
    pcl::PointCloud<pcl::PointXYZRGBL> input;
    f3ps::loadPCDFile(file, input);
    clean_input(input, o);
    pcl::PointCloud<pcl::PointXYZRGBA> cloud;
    pcl::copyPointCloud(input, cloud);
    std::vector<int> devs; for (int d = 0; d < slabs; ++d) devs.push_back(d);
    f3ps_host::SlabRun run(devs);
    if (!run.ok()) { fprintf(stderr, "error: slab mode on %d GPUs: %s\n", slabs, run.init_error().c_str()); return 2; }
    f3ps_host::SlabParams sp;
    sp.voxel_res = o.voxel_resolution; sp.seed_res = o.seed_resolution; sp.color_imp = o.color_importance; sp.spatial_imp = o.spatial_importance;
    sp.normal_imp = o.normal_importance; sp.use_transform = o.disable_transform ? 0 : 1; sp.fold_negative_z = 0;
    sp.color_distance = o.rgb ? F3PS_RGB_EUCL : F3PS_LAB_CIEDE00; sp.geometric_distance = o.cvx ? F3PS_CONVEX_NORMALS_DIFF : F3PS_NORMALS_DIFF;
    sp.merging = o.ml ? F3PS_MANUAL_LAMBDA : (o.eq ? F3PS_EQUALIZATION : F3PS_ADAPTIVE_LAMBDA);
    sp.lambda = (o.ml && o.lambda != 0) ? o.lambda : 0.5f; sp.bins = (o.eq && o.bin_num != 0) ? o.bin_num : 500; sp.threshold = o.thresh;
    const int64_t n = (int64_t)cloud.size();
    std::vector<f3ps_host::SlabShare> shares((size_t)slabs);
    for (int r = 0; r < slabs; ++r) {
        const int64_t lo = n * r / slabs, hi = n * (r + 1) / slabs;
        shares[(size_t)r].points = cloud.points.data() + lo; shares[(size_t)r].n = hi - lo; shares[(size_t)r].stride = 32;
    }
    auto t0 = std::chrono::steady_clock::now();
    if (run.run(shares, sp)) {
        for (int r = 0; r < slabs; ++r) if (!run.info(r).error.empty()) fprintf(stderr, "error: slab rank %d: %s\n", r, run.info(r).error.c_str());
        return 2;
    }
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    f3ps_ctx* h = run.handle(0);
    f3ps_counts c; f3ps_get_counts(h, &c);
    printf("Loading pointcloud from PCD file '%s'...\nFound %d supervoxels\n", file.c_str(), c.n_supervoxels);
    if (o.verbose) {
        std::vector<uint32_t> ab(2 * (size_t)c.n_merges), left(2 * (size_t)c.n_merges); std::vector<float> w((size_t)c.n_merges);
        if (c.n_merges) f3ps_get_merge_log(h, ab.data(), w.data(), left.data(), (int64_t)c.n_merges);
        for (int m = 0; m < c.n_merges; ++m) printf("left: %de/%dp - w: %f - [%d, %d]...OK\n", left[2 * m], left[2 * m + 1], w[(size_t)m], ab[2 * m], ab[2 * m + 1]);
    }
    printf("Clustering complete: %lld points -> %d merges -> %d segments over %d voxels in %.3f ms (%d GPUs, slab mode over NCCL)\n",
           (long long)n, c.n_merges, c.n_segments, c.n_labeled, ms, slabs);
    std::map<std::string, float> worst; std::vector<std::string> order;
    for (int r = 0; r < slabs; ++r)
        for (auto& kv : run.info(r).stage_ms) { if (!worst.count(kv.first)) order.push_back(kv.first); worst[kv.first] = std::max(worst[kv.first], kv.second); }
    printf("  stage ms (max over ranks):");
    for (auto& k : order) printf(" %s %.3f", k.c_str(), worst[k]);
    printf("\n  voxels %lld, exchanged %.1f MB (rank 0)\n", (long long)run.info(0).V, (double)run.info(0).bytes_exchanged / 1e6);
    if (!o.out.empty()) {
        pcl::PointCloud<pcl::PointXYZL> labeled;
        std::vector<float> xyz(3 * (size_t)c.n_labeled); std::vector<uint32_t> lab((size_t)c.n_labeled), vox((size_t)c.n_labeled);
        if (c.n_labeled) f3ps_get_labeled_cloud(h, xyz.data(), lab.data(), vox.data(), c.n_labeled);
        labeled.points.resize((size_t)c.n_labeled);
        for (int i = 0; i < c.n_labeled; ++i) { auto& q = labeled.points[(size_t)i]; q.x = xyz[3 * (size_t)i]; q.y = xyz[3 * (size_t)i + 1]; q.z = xyz[3 * (size_t)i + 2]; q.label = lab[(size_t)i]; }
        labeled.width = (uint32_t)c.n_labeled; labeled.height = 1;
        f3ps::savePCDFileASCII(o.out, labeled);
    }
    return 0;
}

int main(int argc, char** argv) {
    if (argc < 3) { usage(argv[0]); return 1; }
    Options o;
    o.verbose = find_switch(argc, argv, "--V");
    o.disable_transform = find_switch(argc, argv, "--NT");
    o.facade = find_switch(argc, argv, "--facade");
    std::vector<std::string> file_list; std::string path;
    if (find_switch(argc, argv, "-d")) {
        parse(argc, argv, "-d", path);
        if (!std::filesystem::exists(path) || !std::filesystem::is_directory(path)) { fprintf(stderr, "Specified directory doesn't exists or can't be opened\n"); return 1; }
        for (auto& e : std::filesystem::recursive_directory_iterator(path))
            if (e.is_regular_file() && e.path().extension() == ".pcd") file_list.push_back(e.path().string());
        printf("Found %zu files\n", file_list.size());
    } else if (find_switch(argc, argv, "-p")) { parse(argc, argv, "-p", path); file_list.push_back(path); }
    else { fprintf(stderr, "No input file or directory specified\n"); return 1; }
    o.thresh_specified = find_switch(argc, argv, "-t");
    if (o.thresh_specified) parse(argc, argv, "-t", o.thresh);
    else if (find_switch(argc, argv, "--facade")) { fprintf(stderr, "the threshold sweep runs on the direct path: drop --facade or pass -t <threshold>\n"); return 1; }
    parse(argc, argv, "-v", o.voxel_resolution); parse(argc, argv, "-s", o.seed_resolution);
    parse(argc, argv, "-c", o.color_importance); parse(argc, argv, "-z", o.spatial_importance); parse(argc, argv, "-n", o.normal_importance);
    o.rgb = find_switch(argc, argv, "--RGB"); o.cvx = find_switch(argc, argv, "--CVX");
    o.ml = find_switch(argc, argv, "--ML"); o.al = find_switch(argc, argv, "--AL"); o.eq = find_switch(argc, argv, "--EQ");
    if (!(o.ml || o.al || o.eq)) o.al = true;
    else if (!(o.ml ^ o.al ^ o.eq)) { fprintf(stderr, "Only one parameter between --ML --AL and --EQ can be specified at a time\n"); return 1; }   // XOR quirk kept (:280)
    if (o.ml) parse(argc, argv, "--ML", o.lambda);
    if (o.eq) parse(argc, argv, "--EQ", o.bin_num);
    parse(argc, argv, "-o", o.out);
    o.remove_label = find_switch(argc, argv, "-r");
    if (o.remove_label) { int r = 0; parse(argc, argv, "-r", r); o.label_to_be_removed = (uint32_t)r; }
    if (find_switch(argc, argv, "-f")) parse(argc, argv, "-f", o.test_filename);
    o.eval = !find_switch(argc, argv, "--no-eval");
    std::string levels;
    if (parse(argc, argv, "--levels", levels)) {
        for (const char* c = levels.c_str(); *c;) {
            char* end = nullptr;
            o.levels.push_back(strtof(c, &end));
            if (end == c || (*end && *end != ',')) { fprintf(stderr, "--levels takes comma-separated thresholds\n"); return 1; }
            c = *end ? end + 1 : end;
        }
        if (o.levels.empty()) { fprintf(stderr, "--levels takes comma-separated thresholds\n"); return 1; }
    }
    parse(argc, argv, "--point-labels", o.point_labels);
    parse(argc, argv, "--segments", o.segments);
    if ((!o.levels.empty() || !o.point_labels.empty() || !o.segments.empty()) && (o.facade || find_switch(argc, argv, "--slabs"))) {
        fprintf(stderr, "--levels, --point-labels and --segments run on the direct path of one GPU per file: drop --facade / --slabs\n"); return 1;
    }
    int gpus = 1; parse(argc, argv, "--gpus", gpus); gpus = std::max(1, gpus);
    int inflight = 8; parse(argc, argv, "--inflight", inflight); inflight = std::max(1, inflight);
    setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);                     // before the CUDA context exists (see f3ps_create)
    int slabs = 0; parse(argc, argv, "--slabs", slabs);
    if (slabs > 0) {
        if (file_list.size() != 1 || !o.thresh_specified || o.facade) { fprintf(stderr, "--slabs needs one input file (-p) and a threshold (-t)\n"); return 1; }
        try { return run_slabs(file_list[0], o, slabs); } catch (const std::exception& e) { fprintf(stderr, "error: %s\n", e.what()); return 2; }
    }
    int rc = 0;
    std::vector<std::string> reports(file_list.size());
    std::vector<FileScores> scores(file_list.size());
    try {
        if (file_list.size() <= 1 || o.facade) { for (size_t i = 0; i < file_list.size(); ++i) rc |= process_file(file_list[i], o, 0, reports[i], nullptr, scores[i], file_list.size() > 1); }
        else {
            // -d sweep: files are independent (fresh SupervoxelClustering + Clustering per file in the reference, :348,408).
            // `inflight` frames per GPU, each on its own handle / stream / host thread; reports are printed in file order.
            std::mutex emu; std::string first_error;
            if (o.thresh_specified && o.out.empty() && o.levels.empty() && o.point_labels.empty() && o.segments.empty()) {
                // groups of `inflight` files per GPU: front stages per file, ONE merge launch per group (-o, --levels,
                // --point-labels and --segments need the per-file path below)
                std::vector<std::vector<size_t>> share((size_t)gpus);
                for (size_t i = 0; i < file_list.size(); ++i) share[i % (size_t)gpus].push_back(i);
                std::vector<std::thread> th;
                for (int gdev = 0; gdev < gpus; ++gdev)
                    th.emplace_back([&, gdev]() { sweep_device(share[(size_t)gdev], file_list, o, gdev, std::min(inflight, 96), reports, scores, first_error, emu); });
                for (auto& t : th) t.join();
            } else {
                const int workers = (int)std::min<size_t>((size_t)gpus * inflight, file_list.size());
                const bool blocking = workers > (int)std::max(1u, std::thread::hardware_concurrency() / 2);
                std::vector<std::thread> th;
                for (int w = 0; w < workers; ++w) th.emplace_back([&, w]() {
                    try {
                        f3ps::Handle h(w % gpus);
                        f3ps_set_blocking_wait(h.get(), blocking ? 1 : 0);
                        for (size_t i = w; i < file_list.size(); i += workers) process_file(file_list[i], o, w % gpus, reports[i], &h, scores[i], true);
                    } catch (const std::exception& e) { std::lock_guard<std::mutex> g(emu); if (first_error.empty()) first_error = e.what(); }
                });
                for (auto& t : th) t.join();
            }
            if (!first_error.empty()) throw std::runtime_error(first_error);
        }
        for (auto& r : reports) fputs(r.c_str(), stdout);
        if (o.eval) { manage_all_performances(scores, o.test_filename); print_best_performances(scores); }
    } catch (const std::exception& e) { fprintf(stderr, "error: %s\n", e.what()); return 2; }
    return rc;
}
