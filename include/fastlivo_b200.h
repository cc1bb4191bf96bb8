/* fastlivo_b200 -- C ABI of the B200-native FAST-LIVO measurement/ESKF hot path.
 *
 * Plain C, plain pointers and sizes, no torch / Eigen / PCL types.  Every entry
 * point cites the reference code it replaces (paths relative to the reference
 * tree hku-mars/FAST-LIVO @ dcebf84).  INTEGRATION.md shows the bindings a
 * maintainer of the reference adds on its side.
 *
 * Conventions
 *   - all pointers are HOST pointers owned by the caller for the duration of
 *     the call only; the library copies.  The opaque handle owns all device
 *     memory, one CUDA stream and (optionally) one NCCL communicator.
 *   - matrices are row-major doubles; rotations are 3x3 row-major.
 *   - every function returns an int status: FLB_OK (0) or a negative FLB_ERR_*;
 *     nothing throws or aborts.  flb_last_error() gives a message.
 *   - a handle is single-caller; distinct handles are independent.
 *   - there is NO CPU fallback: without a CUDA device flb_create() fails with
 *     FLB_ERR_NO_DEVICE.
 */
#ifndef FASTLIVO_B200_H
#define FASTLIVO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FLB_OK             0
#define FLB_ERR_INVALID   -1  /* bad argument */
#define FLB_ERR_CUDA      -2  /* CUDA runtime error (see flb_last_error) */
#define FLB_ERR_NO_DEVICE -3  /* no usable CUDA device: the product path refuses to run */
#define FLB_ERR_STATE     -4  /* call order: map / scan / image / patches not uploaded */
#define FLB_ERR_NUMERIC   -5  /* singular normal matrix or non-finite state */
#define FLB_ERR_COMM      -6  /* NCCL not available / communicator error */
#define FLB_ERR_TIMEOUT   -7  /* device-side barrier watchdog tripped */

#define FLB_ABI_VERSION 1

typedef struct flb_handle flb_handle;

typedef struct flb_config {
    int    device;           /* CUDA ordinal */
    double cell_size;        /* uniform-grid cell for the device map; <=0 -> 0.6 (2 x filter_size_map) */
    double knn_max_d2;       /* neighbours farther than this never select a point: 5.0,
                                src/laserMapping.cpp:1549; <=0 -> 5.0 */
    double plane_threshold;  /* esti_plane threshold 0.1f, src/laserMapping.cpp:1571; <=0 -> 0.1 */
    int    persistent;       /* 1: one persistent kernel per update (default); 0: kernel-per-pass */
    int    reserved[7];
} flb_config;

/* 18-DoF state == StatesGroup, include/common_lib.h:296-381.
 * cov order [rot, pos, vel, bias_g, bias_a, gravity]. */
typedef struct flb_state18 {
    double rot[9];
    double pos[3];
    double vel[3];
    double bg[3];
    double ba[3];
    double grav[3];
    double cov[324];
} flb_state18;

/* ---- lifetime ------------------------------------------------------------------ */
int         flb_abi_version(void);
int         flb_create(const flb_config* cfg, flb_handle** out);
int         flb_destroy(flb_handle* h);
const char* flb_last_error(const flb_handle* h);   /* h may be NULL: last create error */
/* Run all subsequent work of this handle on an existing CUDA stream (cudaStream_t
 * passed as void*), e.g. torch's current stream.  NULL restores the handle's own. */
int         flb_set_stream(flb_handle* h, void* cuda_stream);
int         flb_synchronize(flb_handle* h);
/* Optional page-locked host buffers.  Upload calls detect page-locked sources (these, cudaHostAlloc or
 * cudaHostRegister memory) and let the copy engine read them directly instead of staging through the
 * handle's own pinned area; such a buffer must then stay unmodified until the next blocking call on the
 * handle (flb_*_update, flb_*_pass, flb_synchronize; for a pipelined frame: the flb_state_download_wait that
 * collects THAT frame's result) returns.  Pageable buffers keep the plain contract: free to reuse as soon as the
 * upload call returns.
 * Uploads never wait for the update that is running: scan, image and patch list each have two device sets, an
 * upload fills the idle one on its own stream and the handle switches sets for everything enqueued afterwards. */
int         flb_host_alloc(flb_handle* h, size_t bytes, void** out);
int         flb_host_free(flb_handle* h, void* p);

/* ---- map: the query half of ikd-Tree -------------------------------------------
 * Replaces KD_TREE::Build (include/ikd-Tree/ikd_Tree.cpp:337-348, called at
 * src/laserMapping.cpp:1411-1419): uploads M map points (float xyz, stride in
 * floats: 3 for packed, 4 for float4, 12 for pcl::PointXYZINormal) and builds the
 * device-resident sorted uniform grid the kNN kernel walks. */
int flb_map_upload(flb_handle* h, const float* xyz, int M, int stride_floats);

/* Device-resident map maintenance (SURVEY.md section 8 row f1): the map follows the reference's ikd-Tree
 * without a per-frame re-upload.
 *   flb_map_add_points  == ikdtree.Add_Points(PointToAdd, true) with downsample_size = filter_size_map
 *                          (map_incremental, src/laserMapping.cpp:692-706; ikd_Tree.cpp:382-457): per
 *                          downsample voxel touched by a new point, only the point closest to the voxel
 *                          centre survives (existing or new); untouched voxels are left alone.  Within a
 *                          few ulps of a voxel boundary the float boxes the reference tests points against
 *                          ([fl(k*ds), fl(fl(k*ds) + ds)) per axis) can overlap or leave a gap, and the
 *                          result depends on the order of the new points: there the reference's rule is
 *                          replayed point by point in submission order, with its exact box test.
 *   flb_map_delete_boxes == ikdtree.Delete_Point_Boxes(cub_needrm) (lasermap_fov_segment,
 *                          src/laserMapping.cpp:363-421; ikd_Tree.cpp:501-521): boxes nb x 6 floats
 *                          (min xyz, max xyz), half-open containment min <= p < max.
 * After either call map indices (flb_knn / flb_lio_export nn_idx) refer to the order flb_map_download
 * returns.  |coordinate / downsample_size| must stay below 2^20. */
int flb_map_add_points(flb_handle* h, const float* world_xyz, int n, int stride_floats, float downsample_size);
int flb_map_delete_boxes(flb_handle* h, const float* boxes, int nb);
int flb_map_size(const flb_handle* h);
int flb_map_download(flb_handle* h, float* xyz, int capacity_points, int* M_out);

/* ---- IMU forward propagation + backward undistortion (SURVEY.md section 8 row f3) ----------------------
 * Replaces ImuProcess::UndistortPcl from src/IMU_Processing.cpp:655 on (called by Process2, :811-849, at
 * src/laserMapping.cpp:1353): per IMU interval the mid-point propagation of attitude / velocity / position
 * and of the 18x18 covariance (cov = F_x cov F_x^T + cov_w, :699-720), the frame-end prediction (:743-758),
 * and the per-point backward motion compensation to the frame end (:778-808).  The LidarMeasureGroup
 * bookkeeping of :613-652 (which points belong to this update, pcl_beg_time, pcl_end_time) stays with the
 * caller.
 *   The device state (flb_state_upload) is state_inout: it is propagated in place (rot_end, pos_end, vel_end,
 *   cov; biases and gravity unchanged), so x_prop and P are on the device for the update that follows
 *   (flb_state_set_prior_enqueue makes it state_propagat, src/laserMapping.cpp:1354).
 *   v_imu: last_imu_ followed by meas.imu (:617-618), times non-decreasing.  carry: the ImuProcess members
 *   that survive from frame to frame (last_lidar_end_time_, acc_s_last, angvel_last), in/out.
 *   pts: n_points lidar-frame points in time order, stride_floats floats apart, x,y,z at [0..2] and the time
 *   offset in ms (PointType::curvature) at [offset_index] (pcl::PointXYZINormal: stride 12, offset_index 9).
 *   out_xyz: n_points x 3 compensated coordinates.  poses_out (optional, capacity n_imu entries of 22 doubles:
 *   offset_time, acc, gyr, vel, pos, rot) receives IMUpose; n_poses_out its length. */
typedef struct flb_imu_sample { double t; double gyr[3]; double acc[3]; } flb_imu_sample;   /* sensor_msgs::Imu */
typedef struct flb_imu_params {
    double cov_gyr[3], cov_acc[3], cov_bias_gyr[3], cov_bias_acc[3];   /* src/IMU_Processing.cpp:15-20, :58-83 */
    double G_m_s2, mean_acc_norm;                                      /* acc * G_m_s2 / mean_acc.norm(), :688 */
    double R_LI[9], t_LI[3];                                           /* Lid_rot_to_IMU, Lid_offset_to_IMU */
} flb_imu_params;
typedef struct flb_imu_carry { double last_lidar_end_time; double acc_s_last[3]; double angvel_last[3]; } flb_imu_carry;
int flb_imu_undistort(flb_handle* h, const flb_imu_params* prm, flb_imu_carry* carry, const flb_imu_sample* v_imu, int n_imu,
                      double pcl_beg_time, double pcl_end_time, const float* pts, int stride_floats, int offset_index,
                      int n_points, float* out_xyz, double* poses_out, int* n_poses_out);

/* ---- scan ------------------------------------------------------------------------
 * feats_down_body (src/laserMapping.cpp:1398-1399): N already-downsampled points in
 * the LiDAR body frame. */
int flb_scan_upload(flb_handle* h, const float* body_xyz, int N, int stride_floats);

/* Exact 5-NN of nq WORLD-frame float queries, KD_TREE::Nearest_Search semantics
 * (include/ikd-Tree/ikd_Tree.cpp:350-380, 843-986, 1291-1295): float32
 * (dx*dx+dy*dy)+dz*dz, ascending order.  idx: nq x 5 indices into the uploaded map,
 * d2: nq x 5.  A query whose 5th neighbour is farther than knn_max_d2 gets
 * idx = -1 / d2 = +inf for the entries beyond knn_max_d2 (the reference rejects such
 * points at src/laserMapping.cpp:1549, so the bounded search is behaviourally identical). */
int flb_knn(flb_handle* h, const float* q_world, int nq, int* idx, float* d2);

/* ---- LIO -------------------------------------------------------------------------- */
typedef struct flb_lio_params {
    double R_LI[9];          /* Lidar_rot_to_IMU     src/laserMapping.cpp:104-105 */
    double t_LI[3];          /* Lidar_offset_to_IMU */
    double laser_point_cov;  /* LASER_POINT_COV      src/laserMapping.cpp:1109 */
    int    max_iteration;    /* NUM_MAX_ITERATIONS: the loop runs iterCount = -1..T-1 (:1506) */
    double conv_rot_deg;     /* 0.01  (:1688); 0 disables the convergence test */
    double conv_pos_cm;      /* 0.015 (:1688) */
} flb_lio_params;

typedef struct flb_lio_report {
    int     passes;
    int     knn_passes;
    int     n_eff_last;      /* effct_feat_num */
    double  res_mean_last;   /* src/laserMapping.cpp:1602 */
    int64_t rows_total;      /* point-to-plane rows assembled over all passes */
    int     converged_last;
    int     status;          /* FLB_OK or FLB_ERR_NUMERIC / FLB_ERR_TIMEOUT raised on device */
} flb_lio_report;

/* Packed normal equations of one pass.  width = 6: live layout [rot, pos]
 * (Hsub, src/laserMapping.cpp:1608-1629); width = 12: IKFoM layout
 * [pos, rot, offset_R_L_I, offset_T_L_I] (h_x, src/laserMapping.cpp:1059-1089). */
typedef struct flb_normal_eq {
    int    width;
    int    n_eff;
    double sum_abs_res;      /* total_residual, :1597 */
    double HTH[144];         /* width x width row-major in the leading entries */
    double HTh[12];
} flb_normal_eq;

/* One pass of the matching loop body src/laserMapping.cpp:1508-1630 at pose (R,p):
 * pointBodyToWorld (:272-286), [kNN (:1543) + esti_plane (common_lib.h:448-493) when
 * rematch], residual + gates (:1573-1584), compaction (:1588-1602), rows (:1608-1629),
 * H^T H / H^T z (:1664-1666).  Also the measurement half of h_share_model (:960-1094)
 * when width = 12 (rematch == ekfom_data.converge, :994). */
int flb_lio_pass(flb_handle* h, const flb_lio_params* prm, const double R[9], const double p[3],
                 int rematch, int width, flb_normal_eq* out);

/* Per-point / per-row products of the LAST flb_lio_pass (any pointer may be NULL):
 *   world_xyz N x 3 float (feats_down_world); nn_idx N x 5 (Nearest_Points as map
 *   indices, -1 = none); nn_d2 N x 5; pabcd N x 4 (cached plane); pd2 N;
 *   selected N (point_selected_surf && res_last<=2, i.e. the row mask);
 *   rows n x width doubles row-major (Hsub or h_x); meas n (meas_vec / h);
 *   sel_idx n (scan index of each compacted row, the order of laserCloudOri). */
int flb_lio_export(flb_handle* h, float* world_xyz, int* nn_idx, float* nn_d2, float* pabcd, float* pd2,
                   uint8_t* selected, double* rows, double* meas, int* sel_idx, int* n_rows);

/* The whole iterated update src/laserMapping.cpp:1504-1733 (control flow: SURVEY.md
 * Appendix A), run on the device without a host round trip per pass.  x: in = state
 * before the update (normally == x_prop), out = updated state and covariance. */
int flb_lio_update(flb_handle* h, const flb_lio_params* prm, flb_state18* x, const flb_state18* x_prop,
                   flb_lio_report* rep);

/* ---- IKFoM-typed LIO update (the `#define USE_IKFOM` estimator) -------------------------
 * state_ikfom (include/use-ikfom.hpp:12-21): pos, rot, offset_R_L_I, offset_T_L_I, vel, bg, ba, grav(S2,
 * |g| = 9.8090).  Quaternions are (x, y, z, w) like Eigen's coeffs(); P is the 23x23 covariance, row-major,
 * in the sub-manifold order above (DOF 23). */
typedef struct flb_state_ikfom {
    double pos[3];
    double rot[4];
    double offset_R_L_I[4];
    double offset_T_L_I[3];
    double vel[3], bg[3], ba[3];
    double grav[3];
    double P[529];
} flb_state_ikfom;

typedef struct flb_ikfom_params {
    double laser_point_cov;  /* R in kf.update_iterated_dyn_share_modified(LASER_POINT_COV, ...), laserMapping.cpp:1484 */
    int    max_iteration;    /* maximum_iter of kf.init_dyn_share(..., NUM_MAX_ITERATIONS, epsi), :1235 */
    double limit[23];        /* epsi (0.001 each, :1233-1234) */
} flb_ikfom_params;

typedef struct flb_ikfom_report {
    int     passes, knn_passes, n_eff_last, converged_last;
    double  res_mean_last;
    int64_t rows_total;
    int     status;
} flb_ikfom_report;

/* esekfom::esekf<state_ikfom,12,input_ikfom>::update_iterated_dyn_share_modified
 * (include/IKFoM_toolkit/esekfom/esekfom.hpp:1619-1928) with h_dyn_share = h_share_model
 * (src/laserMapping.cpp:960-1094), i.e. the block src/laserMapping.cpp:1482-1494, in one device launch:
 * per pass the 12-column rows [n, A, B, C] and h_x^T h_x / h_x^T h, the SO3/S2 re-projection of P, the
 * information-form gain, x [+] dx, the per-component convergence test and, on the last pass, the
 * covariance update.  x: in = x_ (== the propagated state) and P_; out = updated.  Needs the map and the
 * scan uploaded; single GPU, persistent mode. */
int flb_lio_update_ikfom(flb_handle* h, const flb_ikfom_params* prm, flb_state_ikfom* x, flb_ikfom_report* rep);

/* ---- VIO --------------------------------------------------------------------------- */
typedef struct flb_camera {
    int    width, height;
    double fx, fy, cx, cy;   /* vikit PinholeCamera (config/camera_pinhole.yaml) */
    double d[5];             /* radtan; enabled iff |d0| > 1e-7 */
} flb_camera;

typedef struct flb_vio_params {
    double Rcl[9], Pcl[3];   /* camera<-lidar extrinsic, src/laserMapping.cpp:1206 (set_camera2lidar) */
    double R_LI[9], t_LI[3]; /* LidarSelector::set_extrinsic, src/lidar_selection.cpp:35-39 */
    double img_point_cov;    /* src/lidar_selection.cpp:873 */
    int    max_iteration;    /* LidarSelector::NUM_MAX_ITERATIONS */
    float  conv_rot_deg;     /* 0.001f (:883); 0 disables */
    float  conv_pos_cm;      /* 0.001f */
    int    force_all_passes; /* benchmark mode: fixed pass count (no error test, no EKF_end) */
} flb_vio_params;

typedef struct flb_vio_report {
    int     passes[3];       /* index = pyramid level */
    float   last_error[3];
    int64_t rows_total;      /* photometric rows (pixels) assembled over all passes */
    int     skipped_last;    /* patches dropped by the bounds / depth guard in the last pass */
    int     cov_updated;
    int     status;
} flb_vio_report;

typedef struct flb_vio_eq {
    double  HTH[36];
    double  HTz[6];
    float   error;           /* mean squared photometric error, :857 */
    int64_t n_meas;
    int     skipped;
} flb_vio_eq;

/* cv::Mat img of LidarSelector::detect (src/lidar_selection.cpp:1027-1037): gray uint8. */
int flb_image_upload(flb_handle* h, const uint8_t* gray, int width, int height, int stride_bytes);
/* SubSparseMap (include/common_lib.h:263-292) flattened: pos Pn x 3 (Point::pos_),
 * patch Pn x 3 x 64 floats (warpAffine layout, src/lidar_selection.cpp:279-295),
 * search_level Pn. */
int flb_patches_upload(flb_handle* h, const double* pos, const float* patch, const int* search_level, int Pn);
int flb_camera_set(flb_handle* h, const flb_camera* cam);

/* ---- visual-map growth: candidate scoring (SURVEY.md section 8 row f4) -----------------------------------
 * Replaces the first loop of LidarSelector::addSparseMap (src/lidar_selection.cpp:150-168): every point of pg
 * (world frame) is projected into the new frame (T_f_w = [Rcw | Pcw], include/frame.h:89), kept when it lies
 * inside the image with the `border` margin ((patch_size_half+1)*8, :154), scored with vk::shiTomasiScore
 * on the uploaded image (flb_image_upload + flb_camera_set) and takes its grid cell
 * (int(u/grid_size)*grid_n_height + int(v/grid_size), :156) when the score is STRICTLY above the cell's value.
 *   map_value (grid_n_width*grid_n_height floats, grid_n_* = image size / grid_size, :55-56): in = the values
 *   addFromSparseMap left there (:447-455), out = updated.  winner: per cell the index into world_xyz of the
 *   point that took the cell in this call (the reference's add_voxel_points_[cell] / TYPE_POINTCLOUD), -1
 *   otherwise.  Creating the Point / Feature objects for the winners (:174-195) stays with the caller. */
int flb_visual_candidates(flb_handle* h, const double Rcw[9], const double Pcw[3], const float* world_xyz, int n,
                          int stride_floats, int grid_size, int border, float* map_value, int* winner);

/* pcl::VoxelGrid<PointType>::filter on x, y, z (src/laserMapping.cpp:1398-1399 downSizeFilterSurf; src/lidar_selection.cpp:7,
 * :351-352 downSizeFilter): one centroid per occupied leaf, leaves indexed and ordered as PCL does (min_b from the cloud's
 * minimum, idx = ijk . divb_mul, output in ascending idx).  The points of a leaf are summed in float in their INPUT order:
 * PCL's own within-leaf order is that of an unstable std::sort, i.e. unspecified, so this is a defined member of the family
 * of results PCL can produce, not a bit-level reproduction of one PCL build.  out_xyz: up to `capacity` x 3 floats;
 * *n_out = number of occupied leaves.  Uses the handle's scan slot as scratch (upload the scan afterwards).  Blocking. */
int flb_voxel_grid(flb_handle* h, const float* xyz, int n, int stride_floats, float leaf, float* out_xyz, int capacity, int* n_out);

/* ---- device-resident visual map (SURVEY.md section 8 rows f2 and f4) ---------------------------------------
 * The sparse visual map of LidarSelector -- feat_map (unordered_map<VOXEL_KEY, VOXEL_POINTS*>), its Points
 * (include/point.h) with their observation lists of Features (include/feature.h) and the keyframe images those
 * reference -- lives on the device.  Ids (points, features, images) are creation order.  The three calls are the
 * three visual-map steps of LidarSelector::detect (src/lidar_selection.cpp:1027-1080); ComputeJ between them is
 * flb_vio_update / flb_vio_update_enqueue, which consumes the patch list IN PLACE (no host round trip, no
 * flb_patches_upload).  Rcw / Pcw = new_frame_->T_f_w_ (updateFrameState, :905-911); pass NULL for both to take
 * it from the device state with the extrinsics given to flb_vmap_reset.  Single GPU.
 * Needs flb_camera_set and the current frame uploaded with flb_image_upload. */
typedef struct flb_vmap_params {
    int    grid_size;          /* LidarSelector::grid_size (laserMapping.cpp:1198); one patch per grid cell */
    int    ncc_en;             /* :549 */
    double outlier_threshold;  /* :560 */
    double ncc_thre;           /* :552 */
    double Rcl[9], Pcl[3];     /* sparse_map->Rcl / Pcl */
    double R_LI[9], t_LI[3];   /* set_extrinsic(transl, rot), :35-39 */
} flb_vmap_params;
/* clears the map (LidarSelector::init, :41-79) */
int flb_vmap_reset(flb_handle* h, const flb_vmap_params* p);
/* LidarSelector::addFromSparseMap (:346-587).  pg_down: the scan in the world frame after the caller's
 * pcl::VoxelGrid (0.2 m, :7, :351-352), n x stride floats.  Builds sub_sparse_map on the device: positions, warped
 * 3-level reference patches and search levels become the inputs of the next VIO update.  n_selected == NULL:
 * enqueue-only (the count stays on the device); otherwise blocks and returns sub_sparse_map->index.size(). */
int flb_vmap_select(flb_handle* h, const double Rcw[9], const double Pcw[3], const float* pg_down, int n, int stride_floats,
                    int* n_selected);
/* sub_sparse_map of the last flb_vmap_select (blocking; any pointer may be NULL): index (grid cell), point (id),
 * search_levels, propa_errors, voxel_points[i]->pos_, patch (3 x 64 floats each). */
int flb_vmap_selected(flb_handle* h, int capacity, int* n, int* index, int* point, int* search_level, float* error, double* pos,
                      float* patch);
/* LidarSelector::addSparseMap (:142-202): Shi-Tomasi candidate per grid cell over pg (world frame, unfiltered scan),
 * then one new Point + Feature per won cell (AddPoint, :204-230).  Enqueue-only. */
int flb_vmap_grow(flb_handle* h, const double Rcw[9], const double Pcw[3], const float* pg, int n, int stride_floats, int frame_id);
/* LidarSelector::addObservation (:913-965) for the patches of the last flb_vmap_select, with the frame pose AFTER
 * ComputeJ (NULL, NULL = the device state).  Enqueue-only. */
int flb_vmap_add_observations(flb_handle* h, const double Rcw[9], const double Pcw[3], int frame_id);
/* publish_frame_world_rgb (src/laserMapping.cpp:710-745): colour every world point that projects into the current
 * frame with the bilinear BGR sample of LidarSelector::getpixel (src/lidar_selection.cpp:1007-1025).  bgr: the
 * colour frame (img_rgb), 3 bytes per pixel; rgb: n x 3 bytes (r, g, b as the reference stores them); valid[i] = 1
 * for the points the reference pushes into laserCloudWorldRGB (in front of the camera, inside the image), whose order
 * is the input order.  Rcw / Pcw NULL: from the device state (after flb_vmap_reset).  Blocking. */
int flb_colorize(flb_handle* h, const double Rcw[9], const double Pcw[3], const uint8_t* bgr, int stride_bytes, const float* world_xyz, int n,
                 int stride_floats, uint8_t* rgb, uint8_t* valid);
/* sizes (blocking): points, features, keyframe images, patches of the last selection, items appended by the last
 * grow / add_observations call.  Any pointer may be NULL. */
int flb_vmap_counts(flb_handle* h, int* points, int* features, int* images, int* selected, int* last_added);
int flb_vmap_map_value(flb_handle* h, float* out, int capacity);       /* map_value[length] (:356, :455, :162) */
/* the whole map (tests, debugging; blocking): per point pos (3 doubles), value, n_obs, newest-first feature ids
 * (20, -1 padded); per feature px(2) f(3) T_f_w R(9) t(3) = 17 doubles, score, {level, frame id, image slot}. */
int flb_vmap_dump(flb_handle* h, int cap_points, int cap_features, double* pos, float* value, int* n_obs, int* obs20, double* ft_geo17,
                  float* ft_score, int* ft_level_id_img);

/* One measurement pass of LidarSelector::UpdateState (src/lidar_selection.cpp:772-857)
 * at pose (R,p) and pyramid level `level`. */
int flb_vio_pass(flb_handle* h, const flb_vio_params* prm, const double R[9], const double p[3], int level,
                 flb_vio_eq* out);
/* Rows of the LAST flb_vio_pass: z Pn*64 doubles, H_sub Pn*64 x 6 row-major,
 * errors Pn floats (sub_sparse_map->errors). */
int flb_vio_export(flb_handle* h, double* z, double* H_sub, float* errors);

/* LidarSelector::ComputeJ (src/lidar_selection.cpp:967-983): UpdateState (:743-902)
 * for level = 2,1,0, then cov -= G*cov, all on the device. */
int flb_vio_update(flb_handle* h, const flb_vio_params* prm, flb_state18* x, const flb_state18* x_prop,
                   flb_vio_report* rep);
/* float LidarSelector::UpdateState(cv::Mat img, float total_residual, int level) (include/lidar_selection.h:72,
 * src/lidar_selection.cpp:743-902) on its own: the iteration loop of ONE pyramid level starting from *x with
 * last_error = total_residual; returns the level's last_error like the reference (0 when there are no patches).
 * G18x6 (may be NULL): the non-zero block (columns 0..5) of the member G after the call (:874), which the caller's
 * ComputeJ applies as state->cov -= G * state->cov (:980) -- this entry point leaves the covariance alone. */
int flb_vio_update_level(flb_handle* h, const flb_vio_params* prm, int level, float total_residual, flb_state18* x,
                         const flb_state18* x_prop, float* last_error, double* G18x6, flb_vio_report* rep);
/* sub_sparse_map->errors[i] as ComputeJ leaves them (src/lidar_selection.cpp:851: the per-patch errors of the
 * LAST pass executed by the last flb_vio_update / flb_vio_update_enqueue; read by display_keypatch, :995).
 * errors: up to `capacity` floats, patch order. */
int flb_vio_errors(flb_handle* h, float* errors, int capacity);

/* ---- device-resident frame loop (benchmark / pipeline use) ---------------------------
 * Enqueue-only variants: state stays on the device between calls, nothing is copied
 * back until flb_state_download.  flb_frame_enqueue = one LIO update followed by one
 * VIO update whose prior is the LIO posterior (zero-motion propagation). */
int flb_state_upload(flb_handle* h, const flb_state18* x, const flb_state18* x_prop);
int flb_state_download(flb_handle* h, flb_state18* x, flb_lio_report* lio, flb_vio_report* vio);
/* One frame in ONE call (the reference's per-frame work on this path: sync_packages -> LIO update -> VIO update,
 * src/laserMapping.cpp:1269-1460): scan upload, state upload, LIO update, and -- when vprm != NULL -- image upload,
 * patch-list upload (patch_pos == NULL: keep the list already on the device, e.g. one built by flb_vmap_select),
 * state_propagat = state, VIO update; result_slot >= 0 also enqueues the read-back into that slot
 * (flb_state_download_wait collects it).  Everything is enqueue-only. */
typedef struct flb_frame_inputs {
    const float*   scan_xyz;  int n_scan, scan_stride;                 /* feats_down_body, floats per point */
    const uint8_t* gray;      int width, height, stride_bytes;         /* NULL: keep the image on the device */
    const double*  patch_pos; const float* patch; const int* search_level; int Pn;
    const flb_state18* x; const flb_state18* x_prop;
} flb_frame_inputs;
int flb_frame_enqueue(flb_handle* h, const flb_frame_inputs* in, const flb_lio_params* lprm, const flb_vio_params* vprm, int result_slot);
/* Pipelined read-back (two result slots): _enqueue copies the state and both reports of everything enqueued so far and
 * returns at once; _wait blocks on that slot only -- frame k's result is collected while frame k+1 already uploads
 * and runs (uploads never overwrite what an enqueued kernel still reads: stream order, and events for the copy stream). */
int flb_state_download_enqueue(flb_handle* h, int slot);
int flb_state_download_wait(flb_handle* h, int slot, flb_state18* x, flb_lio_report* lio, flb_vio_report* vio);
int flb_lio_update_enqueue(flb_handle* h, const flb_lio_params* prm);
int flb_vio_update_enqueue(flb_handle* h, const flb_vio_params* prm);
/* restore x := x_prop := the state given to the last flb_state_upload (device-side copy) */
int flb_state_reset_enqueue(flb_handle* h);
/* x_prop := x on the device: `state_propagat = state` (src/laserMapping.cpp:1292) with a
 * zero-motion IMU propagation between the LIO and the VIO update */
int flb_state_set_prior_enqueue(flb_handle* h);

/* ---- batched frames (SURVEY.md section 7 H2(iv)) ------------------------------------------------------------
 * B independent frames (own scan, own prior) against the handle's map -- and, for the VIO step, its image and
 * patch list -- advanced together: every pass of the iterated update is ONE launch over all B frames (kernel-per-
 * pass path, blockIdx.y = frame), so the grid is B times a frame's.  One frame's passes are latency-bound at the
 * sizes of BASELINE.json (DESIGN.md section 4); this is the mode in which the kernels run at their throughput
 * (relocalisation against a map, multi-hypothesis tracking, offline batches).  Every frame's result is bit-identical
 * to the same frame run alone through the kernel-per-pass path (flb_config.persistent = 0). */
int flb_batch_begin(flb_handle* h, int B, int max_points_per_frame);
int flb_batch_set_frame(flb_handle* h, int frame, const float* body_xyz, int N, int stride_floats, const flb_state18* x,
                        const flb_state18* x_prop);
int flb_batch_state_reset_enqueue(flb_handle* h);
/* LIO update of every frame, then (vprm != NULL) VIO update with the LIO posterior as prior.  Enqueue-only. */
int flb_batch_update_enqueue(flb_handle* h, const flb_lio_params* lprm, const flb_vio_params* vprm);
int flb_batch_state_download(flb_handle* h, int frame, flb_state18* x, flb_lio_report* lio, flb_vio_report* vio);

/* Per-kernel-family device time of the work enqueued between start and stop,
 * measured with CUDA events on the handle's stream (adds one event pair per launch:
 * use for profiling runs, not for headline timing).  ms[0] = LIO rematch passes,
 * ms[1] = LIO plain passes, ms[2] = VIO passes, ms[3] = solves/finalize; launches[i]
 * the matching launch counts. */
int flb_profile_start(flb_handle* h);
int flb_profile_stop(flb_handle* h, double ms[4], int64_t launches[4]);
/* Device-side pass trace of the persistent kernels (profiling aid; %globaltimer).  After an update,
 * flb_trace_download(which = 0 LIO / 1 VIO) returns microseconds since kernel entry, two per pass:
 * [2k] all blocks arrived at the pass barrier, [2k+1] the leader finished the solve and released. */
int flb_trace_enable(flb_handle* h, int on);
int flb_trace_download(flb_handle* h, int which, double* us, int max_entries, int* n_entries);
/* kernels launched by this handle since creation */
int64_t flb_launch_count(const flb_handle* h);

/* ---- multi-GPU (SURVEY.md §8e) -------------------------------------------------------
 * One process per GPU.  Each rank uploads ITS contiguous shard of the scan points and
 * patches, the full map and image, and identical states; every pass all-reduces the
 * packed normal equations (ncclAllReduce, ncclDouble, ncclSum) and every rank runs
 * the identical solve.  unique_id is the 128-byte ncclUniqueId produced by
 * flb_comm_unique_id on rank 0 and distributed by the caller (e.g. torch.distributed). */
int flb_comm_unique_id(void* unique_id_128b);
int flb_comm_init(flb_handle* h, const void* unique_id_128b, int rank, int world_size);
int flb_comm_destroy(flb_handle* h);

/* Fused NVLink exchange: the B200-idiomatic alternative to the NCCL path.  Inside the persistent update
 * kernel every rank writes its packed sums (leader block) and its VIO per-patch errors (the worker warp that
 * computed each one) straight into every rank's mailbox over NVLink peer memory as self-validating units
 * {payload, exchange tag} -- one store instruction per unit, no separate flag, no system fence, one NVLink
 * traversal per exchange; one kernel per update, no NCCL call, bit-identical results on every rank and to the
 * single-GPU run up to the summation order.  After FLB_ERR_TIMEOUT in this mode the exchange counters of the
 * ranks may differ: repeat flb_p2p_export / flb_p2p_attach on every rank.
 * Each rank: flb_p2p_export() -> 64-byte CUDA IPC handle; gather all handles (rank order) with any host
 * transport; flb_p2p_attach().  One process per GPU, all GPUs NVLink peers; <= 8 ranks. */
int flb_p2p_export(flb_handle* h, void* handle_64b);
int flb_p2p_attach(flb_handle* h, int rank, int world_size, const void* handles_world_x_64b);
int flb_p2p_detach(flb_handle* h);

/* ---- test / tracing aids (not needed by a caller of the path) -------------------------------------------
 * flb_debug_set_packet_epoch: move the pose-packet flag base (wrap-around test).  flb_debug_block_stamps /
 * flb_debug_vio_stamps: per-block %globaltimer stamps of the last traced LIO / VIO update. */
int flb_debug_set_packet_epoch(flb_handle* h, unsigned epoch);
int flb_debug_block_stamps(flb_handle* h, unsigned long long* out, int max_blocks, int* nblocks);
int flb_debug_vio_stamps(flb_handle* h, unsigned long long* out, int max_blocks, int* nblocks, int* words_per_block);
/* flb_debug_scan_order: src_index[i] = index in the caller's scan array of the point at position i of the uploaded
 * (Morton-ordered) scan; capacity >= the scan's point count.  Test aid for the upload's two ordering paths. */
int flb_debug_scan_order(flb_handle* h, int* src_index, int capacity);
/* flb_debug_set_scan_sort: ordering path of the following flb_scan_upload calls -- 0 automatic (by size and by
 * whether the handle's stream is busy), 1 the one-block kernel (scans of <= 25 600 points), 2 the device-wide sort. */
int flb_debug_set_scan_sort(flb_handle* h, int mode);

#ifdef __cplusplus
}
#endif
#endif /* FASTLIVO_B200_H */
