/* f3ps.h -- C ABI of the B200-native supervoxel-plus-merging hot path.
 *
 * Drop-in boundary for the path SURVEY.md section 8 scopes: everything the
 * reference's main() does between "cloud loaded" and "labelled voxel cloud"
 * (/root/reference/src/supervoxel_clustering.cpp:315-367, 408-449), i.e.
 *   pcl::SupervoxelClustering<PointXYZRGBA> (ctor, setters, extract,
 *       getSupervoxelAdjacency)                         supervoxel_clustering.cpp:348-367
 *   Clustering::set_initialstate / cluster / get_*       src/clustering.cpp:605-679
 *   ColorUtilities::mean_color / rgb2lab / lab_ciede00 / rgb_eucl
 *                                                        src/color_utilities.cpp:117-319
 * The C++ facade in include/supervoxel_clustering/ re-creates the reference's
 * class names on top of these calls; a reference maintainer binds them as shown
 * in INTEGRATION.md.
 *
 * Conventions: plain C, opaque handle, int status (0 = ok), no exceptions and no
 * torch / PCL types across the boundary.  One handle owns one CUDA device + stream
 * and all device memory; handles are independent (one per GPU for -d sweeps), a
 * single handle is not thread safe.  Host buffers belong to the caller.
 * There is NO CPU fallback: every entry point fails with F3PS_ERR_CUDA when no
 * device is usable.
 */
#ifndef F3PS_H_
#define F3PS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct f3ps_ctx f3ps_ctx;

enum f3ps_status {
    F3PS_OK = 0,
    F3PS_ERR_INVALID_ARGUMENT = 1, /* std::invalid_argument in the reference (clustering.cpp:579,594) */
    F3PS_ERR_LOGIC = 2,            /* std::logic_error (clustering.cpp:576,591,672) */
    F3PS_ERR_CUDA = 3,             /* CUDA runtime failure / no device */
    F3PS_ERR_CAPACITY = 4,         /* an internal fixed-capacity structure overflowed */
    F3PS_ERR_NOT_CONVERGED = 5     /* expansion fixed point not reached within the sweep budget */
};

/* enums of include/supervoxel_clustering/clustering.h:62-72, same numeric values */
enum f3ps_color_distance { F3PS_LAB_CIEDE00 = 0, F3PS_RGB_EUCL = 1 };
enum f3ps_geometric_distance { F3PS_NORMALS_DIFF = 0, F3PS_CONVEX_NORMALS_DIFF = 1 };
enum f3ps_merging_criterion { F3PS_MANUAL_LAMBDA = 0, F3PS_ADAPTIVE_LAMBDA = 1, F3PS_EQUALIZATION = 2 };

/* stages for f3ps_stage_ms (K1..K7 of SURVEY.md section 2) */
enum f3ps_stage {
    F3PS_STAGE_VOXELIZE = 0, F3PS_STAGE_NEIGHBORS = 1, F3PS_STAGE_NORMALS = 2, F3PS_STAGE_SEEDS = 3,
    F3PS_STAGE_EXPAND = 4, F3PS_STAGE_GRAPH = 5, F3PS_STAGE_MERGE = 6, F3PS_STAGE_TOTAL = 7,
    F3PS_STAGE_MERGE_KERNEL = 8   /* the persistent merge kernel alone (inside F3PS_STAGE_MERGE) */
};

typedef struct f3ps_counts {
    int64_t n_points;      /* N: input points (NaNs included) */
    int64_t n_valid;       /* points that entered a voxel */
    int64_t n_voxels;      /* V */
    int32_t depth;         /* adjacency-octree depth */
    int32_t seed_depth;    /* seed-octree depth */
    int32_t n_seed_cells;  /* occupied seed cells */
    int32_t n_seeds;       /* S0: seeds kept (labels 1..S0) */
    int32_t n_supervoxels; /* S: supervoxels alive after expansion */
    int32_t n_edges;       /* E: initial supervoxel-graph edges (a<b) */
    int32_t n_merges;      /* M: merges performed by the last f3ps_merge */
    int32_t n_segments;    /* regions left */
    int32_t n_edges_left;  /* edges left */
    int32_t rounds;        /* VCCS expansion rounds I */
    int32_t sweeps;        /* total fixed-point sweeps over all rounds */
    int32_t n_labeled;     /* points in the labelled voxel cloud */
    float lambda;          /* lambda in use (adaptive value after f3ps_graph) */
    int32_t max_touched;   /* largest number of edges re-weighted by one merge */
    int64_t fold_steps;    /* voxel steps folded by the merge loop (sum of |b|) */
    int32_t nan_weights;   /* edge weights that evaluated to NaN (regions with < 3 voxels) */
    int32_t merge_path;    /* kernel the last f3ps_merge ran: 0 = none (no supervoxels, or no merge yet), 1 = resident (one SM, weight map in shared memory), 2 = general (also: a resident replay that could not go on, replayed again from the start), 3 = resident with its tables in L2 (graphs too large for an SM), 6 = 1 up to the first merge with more than 928 adjacency entries, then 3 from that state */
} f3ps_counts;

/* ---- life cycle ------------------------------------------------------------ */
/* device: CUDA ordinal.  stream: a cudaStream_t to run on, or NULL for a private one. */
int f3ps_create(int device, void* stream, f3ps_ctx** out);
void f3ps_destroy(f3ps_ctx* ctx);
const char* f3ps_last_error(const f3ps_ctx* ctx);
const char* f3ps_version(void);

/* ---- parameters ------------------------------------------------------------ */
/* SupervoxelClustering(Rv,Rs) + setColor/Spatial/NormalImportance + setUseSingleCameraTransform
 * (supervoxel_clustering.cpp:348-353); fold_negative_z = main()'s z<0 -> |z| (:317-321). */
int f3ps_set_vccs_params(f3ps_ctx* ctx, float voxel_resolution, float seed_resolution, float color_importance,
                         float spatial_importance, float normal_importance, int use_single_camera_transform,
                         int fold_negative_z);
/* Clustering::set_delta_c / set_delta_g / set_merging / set_lambda / set_bins_num
 * (clustering.h:126-137, clustering.cpp:562-597).  Range errors as in the reference. */
int f3ps_set_merge_params(f3ps_ctx* ctx, int color_distance, int geometric_distance, int merging_criterion,
                          float lambda, int bins_num);

/* ---- input ----------------------------------------------------------------- */
/* points: n records of stride_bytes (32 = pcl::PointXYZRGBA {x,y,z,_, b,g,r,a, pad}, 16 = {x,y,z,bgra}).
 * on_device != 0: `points` is device memory valid until the next f3ps_set_input. */
int f3ps_set_input(f3ps_ctx* ctx, const void* points, int64_t n, int stride_bytes, int on_device);

/* ---- stages (each needs the previous one) ------------------------------------ */
int f3ps_voxelize(f3ps_ctx* ctx);   /* K1 OctreePointCloudAdjacency::addPointsFromInputCloud */
int f3ps_neighbors(f3ps_ctx* ctx);  /* K2 computeNeighbors */
int f3ps_normals(f3ps_ctx* ctx);    /* K3 computeVoxelData */
int f3ps_seeds(f3ps_ctx* ctx);      /* K4 selectInitialSupervoxelSeeds */
int f3ps_expand(f3ps_ctx* ctx);     /* K5 expandSupervoxels */
int f3ps_graph(f3ps_ctx* ctx);      /* K6 makeSupervoxels + getSupervoxelAdjacency + set_initialstate + init_weights */
/* K7 Clustering::cluster(threshold): restarts from the initial state.  The same as f3ps_merge_batch of this one handle. */
int f3ps_merge(f3ps_ctx* ctx, float threshold);
/* Grid of K5's cooperative launch.  ctas_per_frame = 0 (default): the whole GPU -- lowest latency for one frame, but
 * cooperative launches of concurrent frames run one at a time.  ctas_per_frame > 0: the grid is capped at that many CTAs (a
 * sweep trades the latency of one frame for more frames side by side).  max_concurrent must be 0; other values, and
 * ctas_per_frame outside 0..296, are F3PS_ERR_INVALID_ARGUMENT.  Same results from every setting. */
int f3ps_set_expand_sharing(f3ps_ctx* ctx, int ctas_per_frame, int max_concurrent);
/* pcl::SupervoxelClustering::refineSupervoxels(num_itr, clusters) (/root/reference/src/supervoxel_clustering.cpp:369-371) on the
 * result of f3ps_expand / f3ps_extract: per iteration SupervoxelHelper::refineNormals (voxel normals from the neighbours of the
 * same supervoxel), reseedSupervoxels (every helper restarts from the voxel nearest to its centroid) and the expansion rounds
 * again from the helpers' current centroids.  Afterwards the per-voxel labels / distances / normals and the supervoxel getters
 * return the refined state; the supervoxel graph is rebuilt by the next f3ps_graph / f3ps_merge.  Calling it before f3ps_expand
 * is F3PS_ERR_LOGIC (PCL: "Supervoxels must be extracted before they can be refined"). */
int f3ps_refine(f3ps_ctx* ctx, int num_itr);
/* which K5 kernel f3ps_expand launches: 0 / 1 = the cooperative grid (lowest latency for one frame: 0.8 ms on a VGA frame, but
 * ~50 SM-ms of mostly barrier waiting; f3ps_set_expand_sharing may cap it), 2 = ONE thread-block cluster per frame
 * (cluster_ctas = 1..16 CTAs of 1024 threads meeting at the hardware cluster barrier; 0 = two voxels per thread, at most 16): the
 * expansion is instruction-bound, so a small cluster does the same work in ~17 SM-ms and leaves the other SMs to the frames next to
 * it -- what directory sweeps use.  Same results from every choice.
 * Replaces pcl::SupervoxelClustering::expandSupervoxels as called from extract() (/root/reference/src/supervoxel_clustering.cpp:357). */
int f3ps_set_expand_kernel(f3ps_ctx* ctx, int which, int cluster_ctas);
/* Clustering::cluster(threshold) for n handles (same device, graphs built) with ONE launch of the resident merge kernel:
 * CTA i replays frame i.  Independent streams share at most 32 hardware queues per context, so a sweep with one merge
 * kernel per stream never overlaps more than 32 of them; a grid has no such limit.  Same results per handle as f3ps_merge;
 * handles whose graph does not fit the resident kernel's shared memory, or whose kernel choice is not 0, are clustered
 * individually, as f3ps_merge would, next to the grids.  A batch of one handle is f3ps_merge, and a grid-able frame left
 * alone (one handle, or the last of more than a grid holds) runs the kernel f3ps_merge would give it, not a one-CTA grid. */
int f3ps_merge_batch(f3ps_ctx** ctxs, int n, float threshold);
/* How the host waits where it needs a size from the device: 0 = spin (lowest latency, the default), 1 = sleep on a
 * blocking event.  Sweeps that keep more frames in flight than there are host cores must use 1. */
int f3ps_set_blocking_wait(f3ps_ctx* ctx, int blocking);
/* which K7 kernel f3ps_merge and f3ps_merge_batch use: 0 = automatic (the resident kernel when the graph fits one SM's shared
 * memory, continued on its L2 variant from the first merge with more than 928 adjacency entries; the L2 variant, with its
 * per-edge / per-region tables in L2, when the graph does not fit but S < 65,535 and E < ~380,000 (16 bytes of shared memory
 * per 32 edges); else the general kernel -- which also replays the whole sequence again when a resident kernel cannot go on:
 * its adjacency pool or stamp range is exhausted, or a merge of the L2 variant has more than 65,534 adjacency entries),
 * 2 = always general, 3 = the L2 variant even when the graph would fit an SM, 4 = 0 with the shared-memory kernel compiled
 * with per-phase cycle counters and the merge trace, 5 = 3 with per-phase cycle counters (f3ps_merge_profile,
 * f3ps_merge_trace); other values, 1 included, are F3PS_ERR_INVALID_ARGUMENT.  Only 0 lets f3ps_merge_batch put a handle into
 * its grid.  All replay the same merge sequence; the switch exists for tests and profiling. */
int f3ps_set_merge_kernel(f3ps_ctx* ctx, int which);
/* Development aid of the resident kernel (kernel choice 4): SM clock values at 32 points of each of 256 consecutive merges,
 * starting at merge `first_merge` of the NEXT f3ps_merge; out (may be NULL to only set the window) receives the last
 * recorded window, 256 x 32 words (slot meaning: f3ps/binding.py merge_trace). */
int f3ps_merge_trace(f3ps_ctx* ctx, int64_t first_merge, uint32_t* out, int64_t capacity_words);
/* SupervoxelClustering::extract + getSupervoxelAdjacency = K1..K5 + supervoxel tables */
int f3ps_extract(f3ps_ctx* ctx);
/* whole path: K1..K7 */
int f3ps_run(f3ps_ctx* ctx, float threshold);
/* blocks until every queued stage is finished */
int f3ps_sync(f3ps_ctx* ctx);

/* Clustering::set_initialstate on caller-supplied supervoxels (clustering.cpp:605-612):
 * voxel arrays (xyz float3, truncated colour 0x00RRGGBB) in the order of each
 * supervoxel's voxels_, supervoxels by ascending label with their voxel ranges,
 * centroid_ (xyz) and normal_ (xyz), and the adjacency multimap in iteration order. */
int f3ps_set_graph(f3ps_ctx* ctx, int64_t n_voxels, const float* voxel_xyz, const uint32_t* voxel_rgba,
                   int32_t n_supervoxels, const uint32_t* labels, const int64_t* voxel_offsets,
                   const float* centroids_xyz, const float* normals_xyz,
                   int64_t n_adjacency, const uint32_t* adjacency_pairs);

/* ---- results (copy out; capacity in elements of the leading dimension) --------- */
int f3ps_get_counts(f3ps_ctx* ctx, f3ps_counts* out);
int f3ps_get_voxel_keys(f3ps_ctx* ctx, uint32_t* keys_xyz /*[V][3]*/, int64_t capacity);
int f3ps_get_voxel_centroids(f3ps_ctx* ctx, float* xyz /*[V][3]*/, float* rgb /*[V][3]*/, uint32_t* rgba /*[V]*/,
                             int32_t* count /*[V]*/, int64_t capacity);
int f3ps_get_point_voxel(f3ps_ctx* ctx, int32_t* voxel_of_point /*[N]*/, int64_t capacity);
int f3ps_get_voxel_neighbors(f3ps_ctx* ctx, int32_t* nbr /*[V][27] list order, -1 padded*/, int32_t* nbr_count /*[V]*/,
                             int64_t capacity);
int f3ps_get_voxel_normals(f3ps_ctx* ctx, float* normal4 /*[V][4]*/, float* curvature /*[V]*/, int64_t capacity);
int f3ps_get_seeds(f3ps_ctx* ctx, int32_t* seed_voxel /*[S0]*/, int64_t capacity);
int f3ps_get_voxel_labels(f3ps_ctx* ctx, uint32_t* label /*[V], 0 = unowned*/, float* distance /*[V]*/, int64_t capacity);
int f3ps_get_supervoxels(f3ps_ctx* ctx, uint32_t* label /*[S]*/, float* centroid_xyz /*[S][3]*/, float* mean_rgb /*[S][3]*/,
                         float* normal4 /*[S][4]*/, int32_t* n_voxels /*[S]*/, int64_t capacity);
/* voxel indices grouped by supervoxel label (ascending), idx order inside = Supervoxel::voxels_ */
int f3ps_get_supervoxel_voxels(f3ps_ctx* ctx, int32_t* voxel_index /*[n_owned]*/, int64_t* offsets /*[S+1]*/,
                               int64_t capacity_voxels, int64_t capacity_supervoxels);
int f3ps_get_adjacency(f3ps_ctx* ctx, uint32_t* pairs /*[2E][2] both directions, sorted*/, int64_t capacity);
int f3ps_get_edges(f3ps_ctx* ctx, uint32_t* ab /*[E][2]*/, float* delta_c, float* delta_g, float* weight, int64_t capacity);
int f3ps_get_cdf(f3ps_ctx* ctx, float* cdf_c /*[bins]*/, float* cdf_g /*[bins]*/, int64_t capacity);
/* the reference's per-merge debug line (clustering.cpp:390-392): edges left, regions left, w, a, b */
int f3ps_get_merge_log(f3ps_ctx* ctx, uint32_t* ab /*[M][2]*/, float* weight /*[M]*/, uint32_t* left /*[M][2]*/, int64_t capacity);
/* Clustering::get_currentstate(): regions (label, centroid, normal, size) and remaining weighted edges in map order */
int f3ps_get_state_regions(f3ps_ctx* ctx, uint32_t* label, float* centroid_xyz, float* normal_xyz, int32_t* n_voxels, int64_t capacity);
int f3ps_get_state_edges(f3ps_ctx* ctx, uint32_t* ab, float* weight, int64_t capacity);
/* ColorUtilities::mean_color of initial region `rank` (ascending-label order), as the edge weights use it */
int f3ps_get_region_mean_color(f3ps_ctx* ctx, int32_t rank, float rgb[3]);
/* Clustering::get_labeled_cloud(): voxel centroids with dense labels 0..K-1 in ascending region label order */
int f3ps_get_labeled_cloud(f3ps_ctx* ctx, float* xyz /*[n][3]*/, uint32_t* label /*[n]*/, uint32_t* voxel_index /*[n]*/, int64_t capacity);
/* per-voxel final segment label (dense, 0xffffffff = unowned) resident on the device; for device consumers */
int f3ps_get_voxel_segments_device(f3ps_ctx* ctx, const uint32_t** device_ptr, int64_t* n);

/* ---- segmentation levels: the segmentation at several thresholds from one merge replay ----
 * Level k is the segmentation f3ps_merge(thresholds[k]) gives: the first m_k merges of the replay, m_k = the first merge log
 * entry whose weight is not below the threshold (M if none).  Labels are dense 0..K-1 per level, in ascending region label
 * order as f3ps_get_labeled_cloud numbers them.  A voxel no supervoxel owns gets 0xffffffff, a phantom leaf its owner's segment;
 * after f3ps_set_graph voxel i is the i-th voxel passed in.  A point gets its voxel's label, 0xffffffff without a voxel.
 * Every merged state has levels: f3ps_merge, f3ps_run and f3ps_merge_batch leave one (their threshold), f3ps_eval_thresholds
 * its last threshold.  The level tables are computed on the first getter call after a merge, on the handle's stream; before
 * any merge the getters return F3PS_ERR_LOGIC. */
/* ONE replay, f3ps_merge(thresholds[n_levels - 1]), recording n_levels levels; the handle is then in exactly the state of that
 * f3ps_merge.  1 <= n_levels <= 256 finite, non-decreasing thresholds, else F3PS_ERR_INVALID_ARGUMENT. */
int f3ps_merge_levels(f3ps_ctx* ctx, const float* thresholds, int n_levels);
/* any output may be NULL; capacity in levels */
int f3ps_get_levels(f3ps_ctx* ctx, int32_t* n_levels, float* thresholds, int32_t* n_merges, int32_t* n_segments, int32_t capacity);
/* labels[L][V] / labels[L][N], level-major; capacity = uint32 elements the buffer holds (>= L*V / L*N).
 * on_device != 0: `labels` is device memory; the write is enqueued on the handle's stream and the call does not wait.
 * on_device == 0: the labels reach the host through a device staging buffer of at most 64 MB, kept by the handle.
 * Point labels are F3PS_ERR_LOGIC after f3ps_set_graph (no input cloud) and in slab mode (after f3ps_slab_set_voxels). */
int f3ps_get_level_voxel_labels(f3ps_ctx* ctx, uint32_t* labels, int64_t capacity, int on_device);
int f3ps_get_level_point_labels(f3ps_ctx* ctx, uint32_t* labels, int64_t capacity, int on_device);

/* ---- segment extraction: the members of every segment of one level, grouped, and one descriptor per segment ----
 * `level` = 0..L-1 indexes the handle's recorded levels (f3ps_get_levels); segments are that level's dense labels 0..K-1, as
 * f3ps_get_level_{voxel,point}_labels number them.  Before any merge: F3PS_ERR_LOGIC; a level out of range or a short buffer:
 * F3PS_ERR_INVALID_ARGUMENT.  The handle keeps the grouping of the last level asked for (points and voxels each) until the next
 * merge, so f3ps_get_segment_info after f3ps_get_segment_points on the same level does not group again.  Grouping a level waits
 * once for its two sizes (members, segments).  on_device != 0: `offsets` / the index array are device memory and the copy into
 * them is enqueued on the handle's stream without a wait; on_device == 0: host memory, read straight from the kept grouping. */
/* points of every segment: offsets[K+1] (offsets[0] = 0, non-decreasing), point_index[offsets[K]] with the points of segment j
 * at [offsets[j], offsets[j+1]) in ascending input order.  Points without a voxel and points whose voxel no supervoxel owns are
 * in no segment.  F3PS_ERR_LOGIC after f3ps_set_graph and in slab mode (as point labels). */
int f3ps_get_segment_points(f3ps_ctx* ctx, int level, int64_t* offsets, int32_t* point_index,
                            int32_t capacity_segments /* >= K+1 */, int64_t capacity_points, int on_device);
/* the same over voxels: voxel indices in ascending order (after f3ps_set_graph voxel i is the i-th voxel passed in); works
 * wherever voxel labels do, slab mode and f3ps_set_graph included */
int f3ps_get_segment_voxels(f3ps_ctx* ctx, int level, int64_t* offsets, int32_t* voxel_index,
                            int32_t capacity_segments, int64_t capacity_voxels, int on_device);
/* One record per segment, host memory, capacity in records (>= K).  Needs the handle's input cloud (F3PS_ERR_LOGIC after
 * f3ps_set_graph and in slab mode); for input on the device it reads the caller's point buffer, which f3ps_set_input requires
 * to stay valid until the next f3ps_set_input.  Sums are reduced in a fixed order (xyz in FP64, rgb in integers): the same
 * bits from every call.  A segment without points (none today: every voxel holds a point) has NaN bounds, centroid and colour. */
typedef struct f3ps_segment_info {
    uint32_t region_label;   /* label of the surviving region (what f3ps_get_state_regions reports at the final level) */
    int32_t  n_voxels;       /* voxels whose level label is this segment (a phantom leaf counts with its owner's) */
    int64_t  n_points;       /* = offsets[j+1] - offsets[j] of f3ps_get_segment_points */
    float    min_xyz[3], max_xyz[3];   /* bounds of its points, coordinates as the path sees them (z<0 -> |z| when folded) */
    float    centroid[3];    /* mean xyz of its points */
    float    mean_rgb[3];    /* mean r, g, b of its points, 0..255 */
} f3ps_segment_info;         /* 64 bytes */
int f3ps_get_segment_info(f3ps_ctx* ctx, int level, f3ps_segment_info* out, int32_t capacity);

/* ---- slab mode: one very large cloud cut into spatial slabs, one per GPU (SURVEY.md section 8e; BASELINE config 5) ----
 * Replaces, for one scan too large or too slow for one device, the same calls as above
 * (pcl::SupervoxelClustering::extract, supervoxel_clustering.cpp:357).  A slab is a contiguous range of the x-major
 * Morton key, i.e. of PCL's leaf index, so every rank's voxels are a contiguous slice of the single-GPU voxel table and
 * all ordered sums keep their order: results are bit-identical to one handle processing the whole cloud.
 * These entry points are the per-rank pieces; the caller issues only the exchanges between them, on the handle's stream
 * (f3ps/slab.py does it with torch.distributed, host/slab_host.cpp with NCCL):
 *   f3ps_set_input(local points) -> f3ps_slab_bbox -> [all-reduce MIN/MAX] -> f3ps_slab_set_frame -> f3ps_slab_keys
 *   -> [all-reduce SUM histogram] -> f3ps_slab_route -> [all-to-all points] -> f3ps_set_input(received, stride 16, on device)
 *   -> f3ps_voxelize -> [all-gather v_local] -> f3ps_slab_set_voxels -> [all-gather voxel slices, in place] -> f3ps_neighbors
 *   -> f3ps_normals (owned slice) -> [all-gather normal slices] -> f3ps_seeds -> f3ps_expand -> f3ps_graph -> f3ps_merge.
 * From f3ps_seeds on every rank works on the whole gathered table; K7 does not shard (strictly serial order over one graph). */
enum f3ps_slab_array_id {
    F3PS_SLAB_VOX_XYZ = 0, F3PS_SLAB_VOX_RGB = 1, F3PS_SLAB_VOX_KEY = 2, F3PS_SLAB_VOX_NORMAL = 3, F3PS_SLAB_VOX_CURV = 4
};
int f3ps_slab_reset(f3ps_ctx* ctx);
int f3ps_slab_bbox(f3ps_ctx* ctx, uint32_t* d_box8);
int f3ps_slab_set_frame(f3ps_ctx* ctx, const uint32_t* d_box8);
/* Morton keys of the local points and the histogram of their top bits into d_hist (1 << top_bits counters, device, top_bits
 * <= 15); the handle keeps the binning for f3ps_slab_route. */
int f3ps_slab_keys(f3ps_ctx* ctx, int top_bits, uint32_t* d_hist);
/* d_hist: the all-reduced histogram (device; may be NULL when world == 1), cut by f3ps_slab_choose_splitters.  Packs the local
 * points as 16-byte records into d_send (capacity: n points), grouped by destination rank; counts[world] = records per rank. */
int f3ps_slab_route(f3ps_ctx* ctx, int world, const uint32_t* d_hist, void* d_send, int64_t* counts);
/* The splitter rule, without a handle or a device: equal-count cuts of hist[n_bins] (bin = key >> shift) into world slabs,
 * each at the first bin boundary at or after its share of the points and never below the cut before it.  out[world - 1]
 * ascend; rank r owns the keys [out[r-1], out[r]). */
int f3ps_slab_choose_splitters(const uint32_t* hist, int n_bins, int world, int shift, uint64_t* out);
/* device arrays the caller exchanges in place: pointer, elements (V), bytes per element */
int f3ps_slab_array(f3ps_ctx* ctx, int which, void** ptr, int64_t* n, int* elem_bytes);
/* Right after f3ps_voxelize on the received points: grows the voxel tables to the whole cloud's n_voxels (< 2^30) and moves
 * this rank's v_local voxels to [own_begin, own_begin + v_local), the slice it owns; the caller fills the other slices. */
int f3ps_slab_set_voxels(f3ps_ctx* ctx, int64_t n_voxels, int64_t own_begin);

/* ---- "next" row f1: the auto-threshold sweep ------------------------------------------------------------------------
 * Clustering::all_thresh (clustering.cpp:691-729) with Testing::eval_performance (testing.cpp:239-362) from ONE merge replay:
 * truth_label[V] = ground-truth label of every voxel (the labelled voxel cloud main() builds, supervoxel_clustering.cpp:387-400),
 * thresholds[n] ascending (main(): 0.8 .. 1 in float steps of 0.005); perf[n] = performanceSet (testing.h:68-75) per threshold,
 * n_segments[n] / n_merges_at[n] (optional) = regions left / merges done at each threshold.  Leaves the handle in the state
 * of f3ps_merge(thresholds[n-1]).  Intersections by exact xyz become equality of the voxel index: truth_label[v] = 0xffffffff
 * marks a voxel without a ground-truth point at its xyz, extra_truth_label[n_extra] lists the labels of ground-truth points
 * that are not voxels of the segmentation (after f3ps_set_graph only owned voxels are known to the handle). */
typedef struct f3ps_performance { float voi, precision, recall, fscore, wov, fpr, fnr; } f3ps_performance;
int f3ps_eval_thresholds(f3ps_ctx* ctx, const uint32_t* truth_label, int64_t n_voxels, const uint32_t* extra_truth_label, int64_t n_extra,
                         const float* thresholds, int n_thresholds, f3ps_performance* perf, int32_t* n_segments, int32_t* n_merges_at);

/* Testing(segm, truth).eval_performance() (testing.cpp:62-146, 239-406) for ONE pair of labelled clouds: the caller pairs the
 * points by exact xyz (as count_intersect does) and passes, per segmentation point, its dense segment label seg[i] < n_seg and
 * the dense ground-truth label of the point at the same xyz, truth[i] < n_truth, or n_truth when there is none; truth_sizes[j] =
 * points of ground-truth segment j, n_truth_points = truth->size().  The contingency table is counted on the device. */
int f3ps_eval_label_pairs(f3ps_ctx* ctx, const uint32_t* seg, const uint32_t* truth, int64_t n_pairs, int32_t n_seg, int32_t n_truth,
                          const uint64_t* truth_sizes, int64_t n_truth_points, f3ps_performance* perf);

/* CUDA-event time of the last run of a stage, ms (valid after f3ps_sync) */
int f3ps_stage_ms(f3ps_ctx* ctx, int stage, float* ms);
/* Profiling aid: SM cycles (clock64) the last f3ps_merge spent per phase, and event counts.
 * General kernel: [0..4] argmin, fold||edge scan, ordering, re-weighting, tie stamps (thread 0).
 * Resident kernel (kernel choice 4, or 5 for the variant with its tables in L2), worker thread 0: [0..6] rescan + publish, wait at
 * S1 + head, adjacency entries + marks, dedupe + speculative colour deltas, wait for the fold, weights + stamps + keys, wait at W4;
 * [7] cycles inside merges with more than 928 adjacency entries (choice 5), [20..23] their four looped phases (entries + marks +
 * guess, dedupe + colour + wait for the fold, weights + classes + list, stamps + keys + clear);  [8..10] / [28..30] cycles / merges by
 * adjacency entries (<= 32, <= 128, more), [11] / [31] the same for merges with more than 928;  [12..15] colour-mean warp: wait for the
 * voxels, fold, Lab + publish, wait for the next head;  [16..19] covariance warp: same with centroid + eigen-solve;  [24] wrong colour
 * guesses, [25] colour-distance evaluations, [27] adjacency entries in total.  f3ps/binding.py merge_profile() names them. */
int f3ps_merge_profile(f3ps_ctx* ctx, uint64_t cycles[32]);
/* nanoseconds the expansion kernel spent per phase: init, sweeps, count, scan, fill, centroid fold, tail, (spare) */
int f3ps_expand_profile(f3ps_ctx* ctx, uint64_t ns[8]);
/* number of kernel launches issued by this handle since creation (bench.py's gpu_launches) */
int64_t f3ps_launch_count(const f3ps_ctx* ctx);

/* metric kernels on the device, for known-answer tests (ColorUtilities::rgb2lab / lab_ciede00 / rgb_eucl):
 * n colour pairs in, n values out; host pointers. */
int f3ps_test_rgb2lab(f3ps_ctx* ctx, const float* rgb255 /*[n][3]*/, float* lab /*[n][3]*/, int64_t n);
int f3ps_test_lab_ciede00(f3ps_ctx* ctx, const float* lab1, const float* lab2, float* out, int64_t n);
int f3ps_test_rgb_eucl(f3ps_ctx* ctx, const float* rgb1, const float* rgb2, float* out, int64_t n);
/* radix sort self-test: sorts (key,value) pairs on the device, stable */
int f3ps_test_sort_pairs(f3ps_ctx* ctx, uint64_t* keys, uint32_t* values, int64_t n, int key_bits);

#ifdef __cplusplus
}
#endif
#endif /* F3PS_H_ */
