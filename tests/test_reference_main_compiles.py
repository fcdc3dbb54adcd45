"""Drop-in check of the boundary (SURVEY.md section 8b): the reference's OWN main() hot-path lines --
/root/reference/src/supervoxel_clustering.cpp:303-457, from "Loading pointcloud" through extract / refineSupervoxels /
getSupervoxelAdjacencyList / label2color / set_initialstate / all_thresh / best_thresh / cluster / get_currentstate /
Testing::eval_performance -- are compiled VERBATIM against include/supervoxel_clustering/ (g++ -fsyntax-only).  Only what the
reference takes from Boost and from PCL's console / io modules is replaced by compile-only stand-ins; every class and method
on the path must exist in the shim with a signature those lines accept.  Runs when F3PS_REFERENCE_DIR names a checkout of the
original project."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(os.environ.get("F3PS_REFERENCE_DIR", ""), "src", "supervoxel_clustering.cpp")

HARNESS = r'''
#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <map>
#include <memory>
#include <string>
#include <vector>
#include "supervoxel_clustering/clustering.h"
#include "supervoxel_clustering/testing.h"
// ---- what the reference pulls in from Boost / PCL beyond the shim: compile-only stand-ins ----
namespace boost {
using std::make_shared;
struct setS {}; struct undirectedS {};
template <class A, class B, class C, class D, class E> struct adjacency_list { typedef void* vertex_descriptor; typedef void* edge_descriptor; };
}
namespace pcl {
namespace console { inline void print_info(const char*, ...) {} inline void print_debug(const char*, ...) {} inline void print_error(const char*, ...) {} inline void print_highlight(const char*, ...) {} }
namespace io { template <class CloudT> int loadPCDFile(const std::string&, CloudT&) { return 0; } }
template <class T> bool isNan(T v) { return v != v; }
}
namespace f3ps {   // the adapter a maintainer writes for the BGL graph (INTEGRATION.md); found by argument-dependent lookup
template <class A, class B, class C, class D, class E>
void f3ps_copy_adjacency_list(const VoxelAdjacencyList&, boost::adjacency_list<A, B, C, D, E>&) {}
}
using namespace boost;
using namespace pcl;
typedef PointXYZRGBA PointT;                    // src/supervoxel_clustering.cpp:67-74
typedef PointCloud<PointT> PointCloudT;
typedef PointNormal PointNT;
typedef PointCloud<PointNT> PointNCloudT;
typedef PointXYZL PointLT;
typedef PointCloud<PointLT> PointLCloudT;
typedef PointXYZRGBL PointLCT;
typedef PointCloud<PointLCT> PointLCCloudT;

// the locals main() declares before the loop (:185-302), as parameters
int reference_main_body(std::vector<std::string> file_list, bool disable_transform, bool thresh_specified, float thresh, float voxel_resolution,
                        float seed_resolution, float color_importance, float spatial_importance, float normal_importance,
                        bool rgb_color_space_specified, bool convexity_specified, bool manual_lambda_specified, bool adapt_lambda_specified,
                        bool equalization_specified, float lambda, int bin_num, bool remove_label, uint32_t label_to_be_removed,
                        float start_thresh, float end_thresh, float step_thresh) {
    PointCloudT::Ptr cloud = make_shared<PointCloudT>();
    PointLCloudT::Ptr truth_cloud = make_shared<PointLCloudT>();
    PointLCCloudT::Ptr input_cloud = make_shared<PointLCCloudT>();
    std::vector<performanceSet> best_performances;
    std::vector<std::map<float, performanceSet> > all_performances;
    std::vector<std::string>::iterator file_it = file_list.begin();
    // ---- /root/reference/src/supervoxel_clustering.cpp:303-457, verbatim ----
'''


@pytest.mark.reference("src/supervoxel_clustering.cpp")
def test_reference_main_hot_path_compiles_against_the_shim(tmp_path):
    lines = open(REF).read().splitlines()
    body = "\n".join(lines[302:457])
    assert "for (; file_it != file_list.end(); ++file_it) {" in lines[302] and "best_performances.push_back(test.eval_performance());" in lines[456]
    for call in ("super.extract(supervoxel_clusters)", "super.refineSupervoxels(3, refined_supervoxel_clusters)", "super.getSupervoxelAdjacencyList(",
                 "Clustering::label2color(", "Clustering::color2label(", "segmentation.set_initialstate(supervoxel_clusters, label_adjacency)",
                 "segmentation.all_thresh(", "segmentation.best_thresh(", "segmentation.cluster(thresh)", "segmentation.get_currentstate()",
                 "segmentation.get_colored_cloud()", "Testing test(segmentation.get_labeled_cloud(), truth_cloud)"):
        assert call in body, call
    src = tmp_path / "reference_main_body.cpp"
    src.write_text(HARNESS + body + "\n    }\n    return 0;\n}\n")
    out = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-I", os.path.join(ROOT, "include"), str(src)], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr[-3000:]
