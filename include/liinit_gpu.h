/* include/liinit_gpu.h -- C-ABI of the B200-native ICP measurement model of LI-Init.
 *
 * The reference has NO plugin / FFI boundary on this path: the code is inlined in
 * main() over file-scope globals (/root/reference/src/laserMapping.cpp:102-125,
 * 957-1134) and the only real API on it is the C++ class KD_TREE
 * (include/ikd-Tree/ikd_Tree.h:165-187). This header is the cut SURVEY.md section 8(b)
 * introduces; every entry point cites the reference lines it replaces.
 *
 * Conventions: extern "C"; opaque context; int return codes (0 = LIINIT_OK, <0 =
 * error, message via liinit_last_error); no exceptions cross the ABI; the caller
 * owns every host buffer, the library owns all device memory; single caller thread
 * (the node's main thread, laserMapping.cpp:891-1238), internally asynchronous on
 * one CUDA stream. Matrices are row-major doubles. Point arrays are float with a
 * caller-given stride in floats: 3 (packed xyz), 4 (float4) or 12 (the 48-byte
 * pcl::PointXYZINormal of include/common_lib.h:37 -- x,y,z are its first floats).
 *
 * There is NO CPU fallback: every compute entry point fails with
 * LIINIT_ERR_CUDA when no sm_100-class device is usable.
 */
#ifndef LIINIT_GPU_H
#define LIINIT_GPU_H

#ifdef __cplusplus
extern "C" {
#endif

#define LIINIT_OK 0
#define LIINIT_ERR_INVALID (-1)   /* bad argument / call order */
#define LIINIT_ERR_CUDA (-2)      /* CUDA runtime error (no device, launch failure, ...) */
#define LIINIT_ERR_CAPACITY (-3)  /* map / scan / hash capacity exceeded */

#define LIINIT_NUM_MATCH_POINTS 5 /* include/common_lib.h:28 */

#define LIINIT_KNN_BRICKS 1
#define LIINIT_KNN_CELLS 2
/* (3, 4, 5 were the hybrid, TMA-fused and warp-per-point searches of round 2: measured slower, removed; profiles/r02, DESIGN.md 3c) */

typedef struct liinit_ctx liinit_ctx;

typedef struct liinit_config {
    float filter_size_map;   /* mapping/filter_size_map (config/avia.yaml:23): map voxel ds; KD_TREE::set_downsample_param (laserMapping.cpp:923) */
    int max_map_points;      /* capacity of the device map (live points); e.g. 50M for BASELINE config 4 */
    int max_scan_points;     /* capacity per scan (replaces the fixed 100000 caps, laserMapping.cpp:108-109,117-119) */
    int device_id;           /* CUDA device ordinal */
    int brick_cells_log2;    /* voxels per brick edge = 1<<this; 0 -> default (3, i.e. brick edge = 8*ds) */
    int hash_capacity_log2;  /* brick hash slots = 1<<this; 0 -> derived from max_map_points */
    int knn_group_lanes;     /* lanes cooperating on one scan point in the lockstep 5-NN kernel: 2, 4, 8, 16 or 32; 0 -> chosen per pass from the frame
                                size (32 lanes up to 14k points, 8 up to 70k, 4 beyond: small frames need the latency, large ones the throughput) */
    float knn_seed_radius_cells; /* first search shell of the 5-NN kernel, in map voxels (radius = this * filter_size_map); 0 -> default (2) */
    int knn_index;           /* how the 5-NN kernel searches the brick hash: LIINIT_KNN_BRICKS (lockstep groups of knn_group_lanes lanes over whole bricks)
                                or LIINIT_KNN_CELLS (thread per scan point over the per-brick cell directory; needs brick_cells_log2 = 3); 0 -> default */
    int reserved[6];
} liinit_config;

/* lifecycle ------------------------------------------------------------------ */
int liinit_create(const liinit_config* cfg, liinit_ctx** out);
int liinit_destroy(liinit_ctx* h);
const char* liinit_last_error(const liinit_ctx* h);   /* h may be NULL: error of the last failed liinit_create */
/* Run on an externally owned stream (cudaStream_t as void*); NULL -> the context's own stream. */
int liinit_set_stream(liinit_ctx* h, void* cuda_stream);

/* map (replaces KD_TREE, include/ikd-Tree/ikd_Tree.h:165-187) ------------------ */
/* KD_TREE::Build (ikd_Tree.cpp:336-347; call site laserMapping.cpp:921-928): replaces the map, no downsampling. */
int liinit_map_build(liinit_ctx* h, const float* xyz, int stride_floats, int n);
/* KD_TREE::Add_Points(points, downsample_on) (ikd_Tree.cpp:381-456; call sites laserMapping.cpp:556-557).
 * added: number of voxels whose content changed (downsample_on) / points appended. */
int liinit_map_add_points(liinit_ctx* h, const float* xyz, int stride_floats, int n, int downsample_on, int* added);
/* KD_TREE::Delete_Point_Boxes (ikd_Tree.cpp:500-520; SURVEY.md row N1 -- the node computes cub_needrm at
 * laserMapping.cpp:260-305 but never passes it on). boxes: nbox x {min x,y,z, max x,y,z} (BoxPointType, ikd_Tree.h:63-66);
 * a point is deleted iff min <= p < max on every axis (:633). deleted: number of points removed. */
int liinit_map_delete_boxes(liinit_ctx* h, const float* boxes, int nbox, int* deleted);
/* Housekeeping the kd-tree does by rebuilding (ikd_Tree.cpp:586-606): slabs abandoned by growth and points removed by box deletes
 * are given back -- live points are re-inserted into a cleared pool, empty bricks leave the hash. Called automatically by
 * liinit_map_add_points / liinit_map_incremental when the pool allocator is in its last quarter and at least half of it is dead;
 * the live set is unchanged. */
int liinit_map_compact(liinit_ctx* h);
/* KD_TREE::validnum / size (ikd_Tree.cpp:71-88,120-137; laserMapping.cpp:932-933,1142): live points. */
int liinit_map_validnum(liinit_ctx* h, int* n);
int liinit_map_size(liinit_ctx* h, int* n);
/* KD_TREE::flatten(Root_Node, out, NOT_RECORD) (ikd_Tree.cpp:1229-1255; laserMapping.cpp:251): live points, packed xyz. */
int liinit_map_download(liinit_ctx* h, float* xyz, int cap_points, int* n);
/* KD_TREE::Nearest_Search for n arbitrary world-frame queries (ikd_Tree.cpp:349-379), max_dist as at laserMapping.cpp:980:
 * squared distance <= max_dist (sic). k must be 5. out_xyz [n*5*3], out_d2 [n*5] (-1 where missing), out_cnt [n]. */
int liinit_map_nearest_search(liinit_ctx* h, const float* q_xyz, int stride_floats, int n, double max_dist,
                              float* out_xyz, float* out_d2, int* out_cnt);
/* KD_TREE::Nearest_Search(point, k, Nearest_Points, Point_Distance, max_dist) (ikd_Tree.cpp:349-379,825-968) for n world-frame
 * queries, any 1 <= k <= LIINIT_KNN_MAX_K and max_dist >= 0 or +INFINITY (the reference's default, ikd_Tree.h:176).
 * out_xyz [n*k*3], out_d2 [n*k], out_cnt [n]: per query the count found, then that many neighbours ascending in PointType_CMP order
 * (ikd_Tree.h:57-60: distances within 1e-10 go by ascending x); d2 = -1 and xyz = 0 past the count.
 *   - d2 is fp32 (dx*dx + dy*dy) + dz*dz without FMA (ikd_Tree.cpp:1273-1277); a point qualifies when d2 <= max_dist (sic, :842),
 *     the float d2 compared with the double max_dist, i.e. with the largest float not above it.
 *   - For max_dist >= 1 or +INFINITY the answer is the exact k nearest live points under that test: the reference's box prune at
 *     max_dist^2 (:827-828) never removes such a point. For 0 <= max_dist < 1 the reference's answer depends on the shape of its
 *     tree; this search applies the point test alone (DESIGN.md section 4, deviations).
 *   - Which of several points tied at exactly the k-th distance is returned is not specified.
 *   - An empty map, a query with a non-finite coordinate or no point within max_dist gives a count of 0. A query far from the map --
 *     also beyond the range brick keys can pack -- still gets its k nearest points when max_dist allows.
 * LIINIT_ERR_INVALID (the context stays usable) for k outside 1..LIINIT_KNN_MAX_K, max_dist NaN or negative, a null pointer, n < 0,
 * or a stride other than 3, 4 or 12. liinit_map_nearest_search and the ICP pass do not use this search. */
#define LIINIT_KNN_MAX_K 32
int liinit_map_knn_search(liinit_ctx* h, const float* q_xyz, int stride_floats, int n, int k, double max_dist,
                          float* out_xyz, float* out_d2, int* out_cnt);
/* Same search with device pointers (queries, outputs), queued on the context's stream with no host synchronisation (as
 * liinit_icp_iterate_device). The host form stages its queries through this one. */
int liinit_map_knn_search_device(liinit_ctx* h, const float* d_q_xyz, int stride_floats, int n, int k, double max_dist,
                                 float* d_out_xyz, float* d_out_d2, int* d_out_cnt);

/* per-scan hot path (replaces laserMapping.cpp:936-1080) ---------------------------- */
/* feats_down_body (laserMapping.cpp:917-919): once per scan; resets selection flags / neighbour lists. */
int liinit_scan_upload(liinit_ctx* h, const float* body_xyz, int stride_floats, int n);
/* Same role, without the staging copy: body_xyz must be page-locked host memory the device can address (cudaHostAlloc,
 * cudaHostRegister, a pinned torch tensor). Nothing is transferred by this call: the search kernel of the next
 * liinit_icp_iterate pass reads the coordinates over PCIe itself and leaves the packed copy in HBM for the later
 * passes of the scan (any other consumer triggers the copy first). The buffer must stay valid and unmodified until
 * that first pass (or liinit_scan_update / liinit_map_incremental / liinit_scan_download_body) has returned; with
 * liinit_icp_iterate_device, until the work queued on the stream has completed.
 * LIINIT_ERR_INVALID when the pointer is not device-addressable page-locked memory. */
int liinit_scan_attach_host(liinit_ctx* h, const float* pinned_body_xyz, int stride_floats, int n);
/* ---- raw-scan front end (SURVEY.md section 8f rows N3, N2): raw points -> undistort -> voxel grid -> resident scan ---- */
/* Stage a raw cloud on the device. time_index: float index of the per-point time offset in MILLISECONDS inside a point
 * (9 = PointType.curvature, src/preprocess.cpp), or -1 when there is none. */
int liinit_raw_upload(liinit_ctx* h, const float* pts, int stride_floats, int time_index, int n);
/* Forward_propagation_without_imu's un-distortion loop (IMU_Processing.hpp:246-266; constant-velocity model, LO mode):
 * omega = state.bias_g (angular velocity), rot_end / vel_end = the PROPAGATED state. In place on the staged cloud. */
int liinit_raw_undistort_cv(liinit_ctx* h, const double omega[3], const double rot_end[9], const double vel_end[3]);
/* propagation_and_undist's back-propagation loop (IMU_Processing.hpp:390-415). poses: the IMUpose table, npose x 22 doubles
 * {offset_time, acc[3], gyr[3], vel[3], pos[3], rot[9]} (Pose6D, common_lib.h:184-199); the state is the propagated one. */
int liinit_raw_undistort_imu(liinit_ctx* h, const double* poses, int npose, const double rot_end[9], const double pos_end[3],
                             const double R_LI[9], const double T_LI[3]);
/* The staged raw cloud as packed xyz (after whatever undistortion ran). */
int liinit_raw_download(liinit_ctx* h, float* xyz, int cap_points, int* n);
/* downSizeFilterSurf.filter (laserMapping.cpp:917-918): voxel grid over the staged cloud -> the resident scan. */
int liinit_raw_downsample(liinit_ctx* h, float leaf_size, int* n_down);
/* Raw (undistorted, not yet downsampled) scan: voxel-grid filter on the device, then the result becomes the resident scan.
 * Replaces downSizeFilterSurf.setInputCloud/filter (laserMapping.cpp:122,823,917-918 = PCL VoxelGrid, leaf = mapping/filter_size_surf)
 * followed by liinit_scan_upload. n_down = feats_down_size. Output order: ascending leaf index, as PCL. */
int liinit_scan_upload_raw(liinit_ctx* h, const float* xyz, int stride_floats, int n, float leaf_size, int* n_down);
/* The resident scan (feats_down_body) as packed xyz. */
int liinit_scan_download_body(liinit_ctx* h, float* xyz, int cap_points, int* n);
/* One ICP pass, laserMapping.cpp:959-1071 + the reduction of :1080.
 *   rot_end, pos_end, R_LI (offset_R_L_I), T_LI (offset_T_L_I): the pose part of StatesGroup (common_lib.h:160-163).
 *   imu_en: 12-column Jacobian (:1054-1062) else 6 columns (:1063-1066).
 *   nearest_search_en: search pass (:978-985) or reuse of stored neighbours and flags (:989-994).
 * Outputs (host): HtH[144] = Hsub^T Hsub (UNWEIGHTED; the reference's R_inv=1000 (:1050) is applied by the
 * caller), Htr[12] = Hsub^T meas_vec with meas = -pd2 (:1070), m = effect_feat_num (:1012-1020).
 * res_sq (optional, may be NULL) = sum of pd2^2 over the selected points. */
int liinit_icp_iterate(liinit_ctx* h, const double rot_end[9], const double pos_end[3], const double R_LI[9],
                       const double T_LI[3], int imu_en, int nearest_search_en, double HtH[144], double Htr[12], int* m,
                       double* res_sq);
/* Same pass, results left on the device: d_out = device pointer to 160 doubles
 * [HtH 144 | Htr 12 | res_sq | m | pad 2], written on the context's stream; no host synchronisation.
 * With a communicator attached (liinit_comm_init) both forms return the SUM over the ranks. */
int liinit_icp_iterate_device(liinit_ctx* h, const double rot_end[9], const double pos_end[3], const double R_LI[9],
                              const double T_LI[3], int imu_en, int nearest_search_en, double* d_out160);
/* laserCloudOri / corr_normvect after compaction (laserMapping.cpp:1013-1020; published at :625-636):
 * ori_xyz [cap*3] body points, normvec [cap*4] = (nx,ny,nz,pd2), order preserved. */
int liinit_scan_download_effect(liinit_ctx* h, float* ori_xyz, float* normvec, int cap_points, int* m);
/* Per-point state of the last pass for parity tests (any pointer may be NULL): world [n*3] (feats_down_world),
 * near_xyz [n*5*3] + near_cnt [n] (Nearest_Points), selected [n] (point_selected_surf), normvec [n*4]. */
int liinit_scan_download_state(liinit_ctx* h, float* world_xyz, float* near_xyz, int* near_cnt, unsigned char* selected,
                               float* normvec);
/* map_incremental (laserMapping.cpp:516-559) with the final state; uses the neighbour lists retained on the
 * device by the last search pass. ds = the node's double filter_size_map_min. n_add / n_no_downsample:
 * sizes of PointToAdd / PointNoNeedDownsample. */
int liinit_map_incremental(liinit_ctx* h, const double rot_end[9], const double pos_end[3], const double R_LI[9],
                           const double T_LI[3], double ds, int flg_EKF_inited, int* n_add, int* n_no_downsample);

/* Test hook: esti_plane<double>(pabcd, points, 0.1) (include/common_lib.h:236-269) of the device for n independent neighbour sets.
 * nb_xyz [n*15] = five xyz per set (f32), pabcd [n*4] = (nx, ny, nz, d), valid [n]. The very function the plane pass calls. */
int liinit_debug_esti_plane(liinit_ctx* h, const float* nb_xyz, int n, double* pabcd, unsigned char* valid);

/* multi-GPU (SURVEY.md section 8e; the reference is single-process, its only parallelism the OpenMP loop laserMapping.cpp:964-968) --------
 * One process (or thread) per GPU, one context each. The map is REPLICATED: every rank makes the same map calls with the same data.
 * The scan is SHARDED: every rank uploads the same whole frame, the library cuts it into nranks equal slots and the search / plane
 * kernels of a rank work on its slot only. The one exchange of the path -- the sum of [HtH 144 | Htr 12 | res_sq | m] over the ranks
 * (one ncclAllReduce of 160 doubles over NVLink on the context's stream) -- happens INSIDE liinit_icp_iterate / _device, so the
 * host-side IESKF loop (liinit_scan_update, liinit_host.h) is unchanged and every rank ends a scan with the same state.
 * liinit_map_incremental and the download hooks first all-gather the per-point results (Nearest_Points copies, flags, normals) of the
 * other ranks' slots, then every rank applies the whole frame's update to its replica: collective calls, same order on every rank.
 * NCCL is loaded with dlopen("libnccl.so.2") when the first of these functions is called; single-GPU use never touches it.
 * How the sum travels: with one process per GPU on an NVLink node, liinit_comm_init maps every rank's 2.6 kB exchange buffer into every
 * process (CUDA IPC) and the LAST BLOCK of the plane kernel does the collective itself -- peer stores of its 160 doubles into every rank's
 * buffer, a system-scope flag, a spin on the other ranks' flags, a rank-ordered sum (bit-identical on every rank): no extra launch, no
 * NCCL kernel. If any rank cannot map its peers (ranks as threads of one process, no peer access) or LIINIT_COMM_MODE=nccl is set, all
 * ranks use ncclAllReduce on the context's stream instead. NCCL always carries the set-up and the all-gathers of per-point results.
 * liinit_map_knn_search / _device are rank-local: each rank answers from its own replica of the map, with no collective.
 * As with any collective: a rank that does not make the call (it returned an error earlier, or died) leaves the others waiting -- the
 * spin in the plane kernel has no time-out, exactly like a pending ncclAllReduce; supervise the ranks from outside. */
#define LIINIT_COMM_ID_BYTES 128
/* ncclGetUniqueId: call on ONE rank, hand the 128 bytes to the others through whatever channel the application has. */
int liinit_comm_unique_id(void* id128);
/* ncclCommInitRank on the context's device; collective over the nranks contexts. LIINIT_ERR_CUDA if NCCL is missing. */
int liinit_comm_init(liinit_ctx* h, const void* id128, int nranks, int rank);
/* This rank's OWN accumulator block of the last pass (before the sum), 160 doubles to the host: lets an application / the bench
 * verify the reduction (sum of the ranks' blocks == what liinit_icp_iterate returned). */
int liinit_comm_last_local(liinit_ctx* h, double* out160);
/* 1 if the accumulators are summed over peer memory inside the plane kernel, 0 if by ncclAllReduce (or no communicator). */
int liinit_comm_mode(liinit_ctx* h, int* peer_memory);
/* nranks / rank of the context and the slot [shard_lo, shard_lo + shard_n) of the resident frame this rank works on. */
int liinit_comm_info(liinit_ctx* h, int* nranks, int* rank, int* shard_lo, int* shard_n);

/* A scan is searched more than once (laserMapping.cpp:1102-1106: rematch after convergence / at the last but one iteration). By default
 * the later search passes of a scan are SEEDED: the five neighbours the previous pass stored still exist in the map (the library tracks
 * every call that can remove a point), so their largest distance from the moved query bounds the new 5th-neighbour distance -- one shell,
 * hardly any inserts, same result bit for bit. enabled = 0 makes every search pass start from scratch (what bench.py times as the metric:
 * the FIRST search pass of a scan). */
int liinit_set_reseed(liinit_ctx* h, int enabled);

/* instrumentation (the reference has none around this loop, SURVEY.md section 5) ---- */
/* Device time in milliseconds of the kernels of the last liinit_icp_iterate* call (CUDA events on the context's
 * stream) and the number of kernel launches it made. */
int liinit_last_pass_timing(liinit_ctx* h, float* kernel_ms, int* launches);
/* Per-kernel device times of the last pass: the 5-NN kernel (0 for a reuse pass) and the plane/Jacobian/reduction kernel. */
int liinit_last_pass_kernel_times(liinit_ctx* h, float* knn_ms, float* plane_ms);
/* The spatial index this context searches (LIINIT_KNN_BRICKS / LIINIT_KNN_CELLS) after defaults were resolved. */
int liinit_knn_index(liinit_ctx* h, int* knn_index);
/* Cumulative number of kernels launched by this context. */
int liinit_launch_count(liinit_ctx* h, long long* launches);
/* Map statistics: bricks in use, hash slots, pool points in use / capacity. */
int liinit_map_stats(liinit_ctx* h, int* bricks, int* hash_slots, long long* pool_used, long long* pool_cap);

#ifdef __cplusplus
}
#endif
#endif /* LIINIT_GPU_H */
