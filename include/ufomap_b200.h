/* ufomap_b200.h -- C ABI of the B200-native UFOMap point-cloud integration path.
 *
 * The reference (UFOMap) has no FFI or plugin layer: its boundary for this path
 * is the C++ class API of libMap (ufo::map::OccupancyMap / OccupancyMapColor,
 * mostly header templates).  Each entry point below names the reference member
 * it stands in for (paths relative to /root/reference/ufomap/include/ufo/map/).
 * The source-compatible C++ facade in include/ufomap_b200/ufomap.hpp forwards to
 * these functions; INTEGRATION.md shows the binding a maintainer would add.
 *
 * Conventions: plain pointers and sizes only; every function returns a
 * ufo_b200_status (0 = OK) unless stated otherwise; a map is bound to one CUDA
 * device and one CUDA stream and is not thread-safe (same as the reference).
 * The library never falls back to a CPU implementation: without a usable
 * device ufo_b200_create fails with UFO_B200_E_CUDA.
 */
#ifndef UFOMAP_B200_H
#define UFOMAP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ufo_b200_map ufo_b200_map;

typedef enum {
	UFO_B200_OK = 0,
	UFO_B200_E_INVALID = 1,     /* bad argument (e.g. depth_levels outside [2,21], octree.h:931-935) */
	UFO_B200_E_CUDA = 2,        /* CUDA runtime error; see ufo_b200_last_error() */
	UFO_B200_E_NOMEM = 3,       /* device pool could not grow */
	UFO_B200_E_UNSUPPORTED = 4  /* documented out-of-scope option (see DESIGN.md) */
} ufo_b200_status;

/* Point buffer layouts accepted by ufo_b200_insert_*: tightly packed AoS. */
typedef enum {
	UFO_B200_XYZ_F64 = 0,     /* double x,y,z             (PointCloud,      point_cloud.h:277) */
	UFO_B200_XYZ_F32 = 1,     /* float  x,y,z             (ROS PointCloud2 payload)            */
	UFO_B200_XYZRGB_F64 = 2,  /* double x,y,z + u8 r,g,b + 5 pad = 32 B (Point3Color, types.h:60-102) */
	UFO_B200_XYZRGB_F32 = 3   /* float  x,y,z + u8 r,g,b + 1 pad = 16 B                        */
} ufo_b200_layout;

/* Constructor arguments of OccupancyMap / OccupancyMapColor (occupancy_map.h:60-63,
 * occupancy_map_base.h:859-876) plus device-side sizing hints. */
typedef struct {
	double resolution;
	uint32_t depth_levels;       /* 2..21, default 16 */
	int32_t automatic_pruning;   /* accepted for API parity; pruning is representational only */
	double occupied_thres;       /* 0.5 */
	double free_thres;           /* 0.5 */
	double prob_hit;             /* 0.7 */
	double prob_miss;            /* 0.4 */
	double clamping_thres_min;   /* 0.1192 */
	double clamping_thres_max;   /* 0.971 */
	int32_t color;               /* 0: OccupancyMap, 1: OccupancyMapColor */
	int32_t device;              /* CUDA device ordinal, -1 = current, -2 = geometry-only handle
	                              * (host indexing / computeRay helpers only, no device state) */
	uint64_t initial_blocks;     /* capacity hint: 4^3-voxel blocks (0 = default) */
	uint64_t initial_bricks;     /* capacity hint: 16^3-voxel bricks (0 = default) */
} ufo_b200_params;

/* Fills *p with the reference's default constructor arguments. */
void ufo_b200_default_params(ufo_b200_params* p);

/* OccupancyMap::OccupancyMap(...)  occupancy_map.h:60-63 */
int ufo_b200_create(const ufo_b200_params* p, ufo_b200_map** out);
void ufo_b200_destroy(ufo_b200_map* m);
const char* ufo_b200_last_error(const ufo_b200_map* m);

/* Run all work of this map on an externally owned CUDA stream (cudaStream_t as
 * void*).  NULL restores the map's own stream. */
int ufo_b200_set_stream(ufo_b200_map* m, void* cuda_stream);

/* insertPointCloud          occupancy_map_base.h:270-327, occupancy_map_color.h:87-160
 * insertPointCloudDiscrete  occupancy_map_base.h:340-417, occupancy_map_color.h:177-267
 *
 * `points` is HOST memory holding n points in `layout`; it is copied before the
 * call returns (the reference takes the cloud by value).  max_range < 0 means
 * unlimited.  depth = insert depth of the free-space rays.  async != 0 returns
 * after the work is enqueued; ufo_b200_wait / ufo_b200_done mirror
 * insertPointCloudWait / insertPointCloudDone (occupancy_map_base.h:430-443).
 * early_stopping != 0 is order-dependent in the reference and is rejected with
 * UFO_B200_E_UNSUPPORTED. */
int ufo_b200_insert_pointcloud(ufo_b200_map* m, const double origin[3], const void* points,
                               size_t n, int layout, double max_range, uint32_t depth,
                               int simple_ray_casting, uint32_t early_stopping, int discrete,
                               int async);

/* Same, but `points` is DEVICE memory on the map's device (no copy is made; the
 * buffer must stay valid until the call's work has finished). */
int ufo_b200_insert_device(ufo_b200_map* m, const double origin[3], const void* d_points,
                           size_t n, int layout, double max_range, uint32_t depth,
                           int simple_ray_casting, uint32_t early_stopping, int discrete,
                           int async);

/* insertPointCloud[Discrete](sensor_origin, cloud, frame_origin, ...) -- the overloads that
 * first move the cloud into the map frame (occupancy_map_base.h:313-327, 403-417;
 * occupancy_map_color.h:146-160, 253-267 -> PointCloudT::transform point_cloud.h:157-166 ->
 * Pose6::transform math/pose6.h:115-125).  frame_pose = {tx, ty, tz, qw, qx, qy, qz}.
 * The transform runs on the device while the points are read (bit-identical to the
 * reference's double arithmetic), so the raw sensor buffer crosses PCIe once. */
int ufo_b200_insert_pointcloud_frame(ufo_b200_map* m, const double origin[3], const void* points,
                                     size_t n, int layout, const double frame_pose[7],
                                     double max_range, uint32_t depth, int simple_ray_casting,
                                     uint32_t early_stopping, int discrete, int async);

/* A sensor_msgs/PointCloud2 buffer exactly as ROS delivers it: n = width*height records of
 * point_step bytes, x/y/z FLOAT32 fields at the given byte offsets, colour bytes at off_r/g/b
 * (for the usual packed "rgb" field at offset o: r = o+2, g = o+1, b = o; -1 = no colour).
 * Replaces rosToUfo (ufomap_ros/ufomap_ros/src/conversions.cpp:77-138): records with a NaN
 * coordinate are skipped, float32 is widened to double, on the device -- the raw buffer is the
 * only thing that crosses PCIe.  frame_pose may be NULL (cloud already in the map frame);
 * otherwise it is the transform the server applies next (server.cpp:116). */
typedef struct ufo_b200_cloud2 {
	const void* data;
	size_t n;
	uint32_t point_step;
	uint32_t off_x, off_y, off_z;
	int32_t off_r, off_g, off_b;
	int32_t on_device; /* != 0: data is device memory on the map's device */
} ufo_b200_cloud2;
int ufo_b200_insert_pointcloud2(ufo_b200_map* m, const double origin[3], const ufo_b200_cloud2* cloud,
                                const double* frame_pose, double max_range, uint32_t depth,
                                int simple_ray_casting, uint32_t early_stopping, int discrete, int async);

/* Host helpers (no device needed).  ufo_b200_transform_points: Pose6::transform of n points of
 * the given layout into out_xyz[n][3].  ufo_b200_pose_from_rpy: Pose6(x, y, z, roll, pitch,
 * yaw) math/pose6.h:71-74 with Quaternion(roll, pitch, yaw) math/quaternion.h:69-93. */
int ufo_b200_transform_points(const double frame_pose[7], const void* points, size_t n, int layout,
                              double* out_xyz);
int ufo_b200_pose_from_rpy(double x, double y, double z, double roll, double pitch, double yaw,
                           double frame_pose[7]);

int ufo_b200_wait(ufo_b200_map* m);           /* insertPointCloudWait */
int ufo_b200_done(ufo_b200_map* m, int* done); /* insertPointCloudDone; never blocks while device work is in flight (completes a scan that ran into a full pool once the device is idle) */

/* Octree::computeRay  octree.h:449-496 -- forward walk, origin voxel included,
 * end voxel excluded.  Writes up to cap codes, *n receives the full count. */
int ufo_b200_compute_ray(const ufo_b200_map* m, const double origin[3], const double end[3],
                         double max_range, uint32_t depth, uint64_t* codes, size_t cap, size_t* n);

/* Octree::toKey / toCode / toCoord  octree.h:299-394, Code <-> Key code.h:183-230 */
int ufo_b200_to_key(const ufo_b200_map* m, const double xyz[3], uint32_t depth, uint32_t key[3]);
int ufo_b200_to_code(const ufo_b200_map* m, const double xyz[3], uint32_t depth, uint64_t* code);
int ufo_b200_key_to_coord(const ufo_b200_map* m, const uint32_t key[3], uint32_t depth,
                          double xyz[3]);
uint64_t ufo_b200_key_to_code(const uint32_t key[3]);
void ufo_b200_code_to_key(uint64_t code, uint32_t key[3]);

/* Node state at (code, depth) with the INTENDED semantics of getOccupancy /
 * getColor / containsFree / containsUnknown (occupancy_map_base.h:599-728; the
 * reference's own Code-based getters read the depth-1 parent, octree.h:974-985).
 * logodds[i]: float log-odds (max over the subtree for depth > 0);
 * flags[i]: bit0 contains_free, bit1 contains_unknown; rgb: 3 bytes per query or NULL.
 * Host pointers. */
int ufo_b200_query(ufo_b200_map* m, const uint64_t* codes, const uint32_t* depths, size_t n,
                   float* logodds, uint8_t* flags, uint8_t* rgb);

/* Dump of the value field: every depth-0 voxel whose payload differs from the
 * default (log-odds 0, colour unset).  Call with codes == NULL to get the count
 * in *n; then with buffers of that capacity (host pointers; rgb may be NULL). */
int ufo_b200_export_leaves(ufo_b200_map* m, uint64_t* codes, float* logodds, uint8_t* rgb,
                           size_t cap, size_t* n);

/* setValueVolume(AABB, occupancy probability, min_depth)  occupancy_map_base.h:492-518 -- the
 * other map writer the mapping server uses (robot clearing server.cpp:152-154, clear_volume
 * service :354).  box6 = the AABB's centre xyz and half_size xyz (geometry/aabb.h:49-70).  Every
 * node of depth min_depth whose cube -- and every ancestor cube -- intersects the box is set to
 * clamp(float(logit(occupancy))) (setOccupancy, :1151-1157), i.e. all voxels below it.
 * min_depth 0..4; colour maps at min_depth 0 only (deeper, the reference also replaces the
 * voxels' colours by the node's mean colour). */
int ufo_b200_set_value_volume(ufo_b200_map* m, const double box6[6], double occupancy, uint32_t min_depth);

/* Octree::write(std::ostream& / filename, bounding_volume, compress = false, min_depth)
 * (octree.h:776-864, writeNodes occupancy_map_base.h:1457-1533): the map as a UFOMap file image
 * -- text header, then the pre-order node stream -- which the reference's Octree::read / the RViz
 * plugin parse; the save_map service of the mapping server (server.cpp:381-392).  box6 (NULL =
 * whole map) and min_depth as for ufo_b200_write_data below.
 * expanded = 0: the canonical tree of the map's value field (a node whose eight children are
 * leaves with equal payload is a leaf).  The reference collapses such nodes itself (updateNode,
 * occupancy_map_base.h:1210-1212 -- logically even with automatic pruning off,
 * octree.h:1060-1066), so this is byte-identical to its own file unless its update order left a
 * collapsible node behind (updateParents stops at the first unchanged aggregate, :1126-1133);
 * then the two files differ in shape only and read back to the same map.  expanded != 0: every
 * octet that was ever touched is written as eight voxels (value-equivalent, larger).
 * ufo_b200_write: *size receives the image size; the image is copied when it fits into cap
 * (call with buf = NULL to size the buffer).  No LZ4. */
int ufo_b200_write(ufo_b200_map* m, const double* box6, uint32_t min_depth, int expanded, void* buf, size_t cap,
                   size_t* size);
int ufo_b200_write_file(ufo_b200_map* m, const char* filename, const double* box6, uint32_t min_depth,
                        int expanded);

/* Octree::writeData(stream, bounding_volume, compress = false, min_depth) (octree.h:885-917): the
 * node stream alone, as ufoToMsg puts it into a UFOMap message
 * (ufomap_ros/ufomap_msgs/include/ufomap_msgs/conversions.h:161-185; the mapping server publishes
 * the changed region at depths 0..publish_depth this way, server.cpp:184-199).  box6 = the
 * fields of a ufo::geometry::AABB: centre xyz, half_size xyz (geometry/aabb.h:49-70; for
 * AABB(min, max) that is half = (max - min) / 2, centre = min + half) or NULL for the whole map:
 * children whose cube misses the box are skipped (intersects(AABB, AABB),
 * collision_checks.cpp:256-264).  Children at min_depth are written as leaves carrying their aggregate
 * (max occupancy, mean colour); min_depth 0..4 is supported.  Canonical tree, see above.
 * *size = 0 when the box misses the map (the reference writes nothing then). */
int ufo_b200_write_data(ufo_b200_map* m, const double* box6, uint32_t min_depth, void* buf, size_t cap,
                        size_t* size);

/* castRay  occupancy_map_base.h:449-486, batched.  The reference's own version does not compile
 * (SURVEY.md G5); this is its intent (DESIGN.md section 8 states it; the CPU checker restates it): max_range < 0 -> the map's
 * diagonal; the ray origin + t * direction, clipped into the map, is walked forward at `depth`;
 * the first occupied node is the hit (hit[i] = 1, codes[i] = its Code), an unknown node ends the
 * ray unless ignore_unknown.  Node state follows the intended getNode semantics of ufo_b200_query. */
int ufo_b200_cast_rays(ufo_b200_map* m, const double* origins, const double* directions, size_t n,
                       int ignore_unknown, double max_range, uint32_t depth, uint64_t* codes, uint8_t* hit);

/* Leaf iteration with state and bounding-volume filters (beginLeaves(occupied, free, unknown,
 * contains = false, min_depth) and its bounding-volume form, occupancy_map_base.h:130-216; validity
 * rule iterator/occupancy_map.h:168-207), as a batch: every node of depth `depth` in the known
 * space whose own state passes the filter (occupied: value > occupied threshold; free: value <
 * free threshold; unknown: in between; an inner node carries the maximum of its subtree) and whose
 * cube intersects the AABB box6 (centre, half size; NULL: everywhere).  codes carry the depth's
 * centre bits; unordered.  A leaf the reference keeps collapsed above `depth` appears as its
 * depth-`depth` cells.  codes == NULL: count only. */
int ufo_b200_export_nodes(ufo_b200_map* m, uint32_t depth, int occupied, int free_space, int unknown, const double* box6,
                          uint64_t* codes, float* logodds, uint8_t* rgb, size_t cap, size_t* n);

/* Octree::write / writeData with compress = true (octree.h:812-917, :1428-1456): the node stream
 * as one LZ4 block (LZ4_compress_fast with acceleration_level when compression_level <= 0, else
 * LZ4_compress_HC), behind the text header with "compressed 1" unless data_only.  liblz4.so.1 is
 * loaded at run time, like the reference links it; UFO_B200_E_UNSUPPORTED if it is absent.
 * *uncompressed_size = what the header's uncompressed_data_size says (writeData's return value). */
int ufo_b200_write_compressed(ufo_b200_map* m, const double* box6, uint32_t min_depth, int data_only,
                              int acceleration_level, int compression_level, void* buf, size_t cap, size_t* size,
                              size_t* uncompressed_size);

/* Octree::readData (octree.h:733-770 -> readNodes, occupancy_map_base.h:1379-1456): merges a node
 * stream -- the body of a UFOMap file, or a UFOMap message the way the ROS layer applies it
 * (msgToUfo, ufomap_msgs/conversions.h:122-134) -- into the map: every leaf of the stream sets all
 * voxels below it to its payload, nodes whose cube misses the AABB box6 (centre, half size; NULL:
 * none) are skipped exactly like the writer skipped them.  The stream must have been written for
 * this map's resolution / depth_levels (the reference clears and resizes otherwise: call
 * ufo_b200_clear_resize first).  compressed != 0: `data` is one LZ4 block of uncompressed_size
 * bytes.  A collapsed non-default node above the brick level is expanded into bricks (at most 2^20
 * per call, else UFO_B200_E_UNSUPPORTED). */
int ufo_b200_read_data(ufo_b200_map* m, const double* box6, const void* data, size_t size, int compressed,
                       size_t uncompressed_size);

/* Sensor model  occupancy_map_base.h:734-773.  out6/in: occupied_thres,
 * free_thres, prob_hit, prob_miss, clamping_thres_min, clamping_thres_max as
 * probabilities (setters) or as stored double log-odds (ufo_b200_sensor_model_logit). */
int ufo_b200_set_sensor_model(ufo_b200_map* m, const double prob6[6]);
/* One sensor-model parameter, the way the reference's setters work (occupancy_map_base.h:748-773:
 * setProbHit / setProbMiss / setClampingThresMin / setClampingThresMax / setOccupiedFreeThres each
 * store toLogit(p) into ONE member and leave the others' stored log-odds untouched).
 * index: 0 occupied_thres, 1 free_thres, 2 prob_hit, 3 prob_miss, 4 clamping_thres_min,
 * 5 clamping_thres_max.  Changing a threshold (0, 1) re-derives the contains_free /
 * contains_unknown flags of every inner node, like the reference's write + read round trip. */
int ufo_b200_set_sensor_model_field(ufo_b200_map* m, int index, double probability);
int ufo_b200_sensor_model_logit(const ufo_b200_map* m, double logit6[6]);

/* min/max change detection  occupancy_map_base.h:792-822 (always enabled). */
int ufo_b200_change_bbox(ufo_b200_map* m, double min_change[3], double max_change[3]);
int ufo_b200_reset_change_bbox(ufo_b200_map* m);

/* Change detection  occupancy_map_base.h:779-790 (enableChangeDetection / resetChangeDetection /
 * changesBegin..changesEnd / numChangedDetected): the set of nodes whose occupancy value changed
 * since the last reset (updateOccupancy returned true, :1070, :1094, :1106).  Recorded per voxel on
 * the device; ufo_b200_changed_codes returns the set at `depth` -- the insert depth the caller
 * used, 0 for the server's default -- as Code values (with the centre bits a Code built from a
 * depth-d Key carries), unordered like the reference's CodeSet.  codes == NULL: count only.
 * enable == 0 pauses the recording and keeps the set, as the reference does: it grows with the map,
 * ufo_b200_changed_codes / ufo_b200_reset_change_detection / ufo_b200_clear act on it as they do
 * while recording, and enabling again resumes recording into it. */
int ufo_b200_enable_change_detection(ufo_b200_map* m, int enable);
int ufo_b200_reset_change_detection(ufo_b200_map* m);
int ufo_b200_changed_codes(ufo_b200_map* m, uint32_t depth, uint64_t* codes, size_t cap, size_t* n);

/* Counters and timings of the most recent insert (waits for it to finish). */
typedef struct {
	uint64_t points;          /* N                                         */
	uint64_t rays;            /* rays cast                                 */
	uint64_t visits;          /* V: voxel visits of the ray walk (only when profiling) */
	uint64_t touched_voxels;  /* U: unique voxels that received an update  */
	uint64_t hit_voxels;      /* U_h                                       */
	uint64_t touched_octets;  /* D_1                                       */
	uint64_t touched_blocks;  /* D_2 (4^3 blocks)                          */
	uint64_t touched_d3;      /* D_3 (8^3 nodes)                           */
	uint64_t touched_bricks;  /* D_4 (16^3 bricks)                         */
	uint64_t upper_nodes;     /* sum of D_l, l >= 5                        */
	uint64_t blocks_in_map;   /* pool occupancy                            */
	uint64_t bricks_in_map;
	uint64_t device_bytes;    /* device memory held by the map             */
	uint64_t regrows;         /* pool growth events during this insert     */
	uint64_t launches;        /* kernels launched by this insert           */
	uint64_t result_bytes;    /* bytes of per-scan counters copied device -> host by this insert */
	uint64_t touched_lines;   /* 128-byte lines of leaf data holding a touched octet (HBM moves whole lines) */
	float ms_total;           /* CUDA-event time of the whole insert (device work) */
	float ms_h2d;
	float ms_points;          /* K1: discretise + hit marking              */
	float ms_rays;            /* K2: ray walk (k_rays)                     */
	float ms_scatter;         /* K2b: record lookup + mask marking (k_scatter) */
	float ms_update;          /* K3: leaf log-odds update + in-block aggregates */
	float ms_propagate;       /* K4: brick + upper-level aggregates        */
} ufo_b200_scan_stats;

int ufo_b200_last_scan_stats(ufo_b200_map* m, ufo_b200_scan_stats* out);
/* Statistics of the most recent scan whose integration is COMPLETE, without waiting for the scan
 * in flight: after an async insert of scan k this returns scan k-1 (its counters were read back
 * when scan k was enqueued).  For callers that stream scans with async = 1 and still want each
 * scan's result.  points == 0 in *out: no scan has completed yet. */
int ufo_b200_completed_scan_stats(ufo_b200_map* m, ufo_b200_scan_stats* out);
/* Octree::clear(resolution, depth_levels)  octree.h:541-560 -- the server's reset service
 * (server.cpp:364-378): empties the map and changes its geometry. */
int ufo_b200_clear_resize(ufo_b200_map* m, double resolution, uint32_t depth_levels);

/* 0: off; 1: per-kernel CUDA-event timing; 2: additionally count ray-walk visits
 * (one extra atomic per ray). */
int ufo_b200_set_profiling(ufo_b200_map* m, int enable);

/* Spatial sharding over several GPUs (SURVEY.md 8(e), variant 1): every rank is given the same
 * scans (broadcast) and keeps only the bricks (16^3-voxel nodes) it owns -- ownership is a hash of
 * the brick key, so the touched space splits evenly wherever the sensor is.  The union of the
 * ranks' value fields is the single-GPU map; no state is exchanged.  Aggregates of depth >= 5 are
 * per rank (partial) in this mode.  Must be called on an empty map.  world <= 1 turns it off. */
int ufo_b200_set_shard(ufo_b200_map* m, uint32_t rank, uint32_t world);

/* Routed multi-GPU mode (SURVEY.md 8(e), variant 2; BASELINE configs #4 "octant shard" and #5
 * "one GPU per sensor with boundary merge").  The reference integrates on one thread
 * (occupancy_map_base.h:270-327); this is the multi-GPU form of the same insertPointCloud:
 * state is owned by space (rank = hash of the 16^3-voxel brick key, as in ufo_b200_set_shard),
 * marking is parallel over rays.  Every rank walks ITS rays -- a slice of one scan, or its own
 * sensor's scan -- and the per-brick free-space masks / hit voxels of bricks another rank owns
 * are written straight into that rank's inbox over NVLink peer memory; the only collective is a
 * barrier between the two calls below (the caller's: e.g. a 4-byte NCCL all-reduce on the map's
 * stream).  Mono maps, insert depth 0, plain (non-discrete) insertion.
 *
 *   ufo_b200_route_setup    allocates this rank's inbox (cap_bricks brick records and cap_hits hit
 *                           voxels per source rank and parity) and returns its device pointer
 *   ufo_b200_ipc_export/_open   cudaIpc handle of that pointer / mapping of a peer's handle, for
 *                           one-process-per-GPU launches (handles travel through the caller's
 *                           control plane, e.g. torch.distributed.all_gather_object)
 *   ufo_b200_route_connect  peer_inboxes[r] = device pointer of rank r's inbox as seen from this
 *                           process (its own for r == rank)
 *   ufo_b200_route_mark     enqueue: H2D, K1, fused walk, forwarding of foreign marks.  self_too != 0:
 *                           the rank's own marks go through its inbox as well, which lets the
 *                           owner apply several sensors one after the other (clamping makes the
 *                           order matter)
 *   -- barrier across the ranks, ordered after route_mark on the map's stream --
 *   ufo_b200_route_apply    enqueue: marks received from sources [first_source, first_source +
 *                           n_sources) -> K3; last != 0 additionally runs the inner-node
 *                           propagation and ends the pass.  One scan split over the ranks:
 *                           route_apply(0, world, 1).  One sensor per rank, merged in sensor order:
 *                           route_apply(s, 1, s == world - 1) for s = 0..world-1.
 * The union of the ranks' value fields equals the single-GPU map (tests/test_gpu_route.py).  Pools
 * do not grow during a routed pass: size the map with initial_bricks. */
int ufo_b200_route_inbox_bytes(uint32_t world, uint32_t cap_bricks, uint32_t cap_hits, size_t* bytes);
int ufo_b200_route_setup(ufo_b200_map* m, uint32_t rank, uint32_t world, uint32_t cap_bricks, uint32_t cap_hits,
                         void** inbox);
int ufo_b200_route_connect(ufo_b200_map* m, void* const* peer_inboxes);
int ufo_b200_route_mark(ufo_b200_map* m, const double origin[3], const void* points, size_t n, int layout,
                        double max_range, int on_device, int self_too);
int ufo_b200_route_apply(ufo_b200_map* m, uint32_t first_source, uint32_t n_sources, int last);
int ufo_b200_ipc_export(void* dev_ptr, void* handle64);
int ufo_b200_ipc_open(const void* handle64, void** dev_ptr);
int ufo_b200_ipc_close(void* dev_ptr);

/* Forget everything (Octree::clear, octree.h:541-560): keeps device pools. */
int ufo_b200_clear(ufo_b200_map* m);

const char* ufo_b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* UFOMAP_B200_H */
