// flb_capi.cu -- the C ABI of include/fastlivo_b200.h over the sm_100a kernels.
// Host side is plain C++ (no Eigen / PCL / torch); the handle owns device memory, three streams (updates; image + patch
// copies; scan copy + ordering -- every input has two device sets, so an upload never waits for the update that is
// running: DESIGN.md section 4.8), CUDA events and an optional NCCL communicator (dlopen'ed lazily).
#include "../../include/fastlivo_b200.h"

#include <cuda_runtime.h>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "flb_kernels.cuh"
#include "flb_vmap.cuh"

using namespace flb;

static_assert(sizeof(flb_state18) == sizeof(State18), "flb_state18 and device State18 must match");
static_assert(sizeof(flb_state_ikfom) == sizeof(StateIkfom), "flb_state_ikfom and device StateIkfom must match");

namespace {

std::string g_create_error;

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = std::max<size_t>(n, 16);
        cudaError_t e = cudaMalloc(&p, want * sizeof(T));
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocMapped);   // mapped: small kernels read / write it in place
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

// Pinned staging area for host->device uploads.  An upload packs the caller's data into it and
// enqueues the copy; `done` marks that copy, and the next user of the same area waits on it (normally
// long complete), so uploads never block on the stream and the caller's buffer is free on return.
struct Staging {
    PinBuf buf;
    cudaEvent_t done = nullptr;
    bool pending = false;
    cudaError_t acquire(size_t bytes, void** out) {
        if (pending) {
            cudaError_t e = cudaEventSynchronize(done);
            if (e != cudaSuccess) return e;
            pending = false;
        }
        cudaError_t e = buf.reserve(bytes);
        if (e != cudaSuccess) return e;
        if (!done) {
            e = cudaEventCreateWithFlags(&done, cudaEventDisableTiming);
            if (e != cudaSuccess) return e;
        }
        *out = buf.p;
        return cudaSuccess;
    }
    cudaError_t mark(cudaStream_t s) {
        cudaError_t e = cudaEventRecord(done, s);
        pending = (e == cudaSuccess);
        return e;
    }
    void release() {
        if (done) cudaEventDestroy(done);
        done = nullptr;
        buf.release();
    }
};

// ---- NCCL through dlopen (no link-time dependency) ----------------------------------
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(ncclUniqueId*) = nullptr;
    int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool load() {
        if (lib) return true;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (lib) break;
        }
        if (!lib) return false;
        GetUniqueId = (int (*)(ncclUniqueId*))dlsym(lib, "ncclGetUniqueId");
        CommInitRank = (int (*)(ncclComm_t*, int, ncclUniqueId, int))dlsym(lib, "ncclCommInitRank");
        CommDestroy = (int (*)(ncclComm_t))dlsym(lib, "ncclCommDestroy");
        AllReduce = (int (*)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t))dlsym(lib, "ncclAllReduce");
        AllGather = (int (*)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t))dlsym(lib, "ncclAllGather");
        GetErrorString = (const char* (*)(int))dlsym(lib, "ncclGetErrorString");
        return GetUniqueId && CommInitRank && CommDestroy && AllReduce && AllGather;
    }
};
NcclApi g_nccl;
constexpr int kNcclInt32 = 2, kNcclFloat32 = 7, kNcclFloat64 = 8, kNcclSum = 0, kNcclMax = 2;  // ncclDataType_t / ncclRedOp_t values (nccl.h)

}  // namespace

struct flb_handle {
    int device = 0;
    flb_config cfg{};
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    // The VIO inputs (image, patch list) are copied on a second stream so that their H2D transfer
    // overlaps the LIO kernel running on `stream`; two events order them against the VIO kernels.
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_vio_inputs = nullptr;   // recorded on copy_stream after the last image / patch copy
    cudaEvent_t ev_vio_done = nullptr;     // recorded on `stream` after the last kernel that reads them
    bool vio_inputs_pending = false, vio_done_pending = false;
    // The image and the host-built patch list are double-buffered like the scan: an upload fills the set that no kernel
    // reads (on copy_stream), then swaps it in; frame k + 1's copies (2 MB at C2) run under frame k's VIO update.
    struct InSlot {
        cudaEvent_t free_ev[2] = {nullptr, nullptr};   // [slot]: recorded on `stream` once every reader of that slot has been enqueued
        bool valid[2] = {false, false};
        int slot = 0;
    } img_slot, patch_slot;
    std::string err;
    int64_t launches = 0;

    // map
    int M = 0;
    GridDesc grid{};
    int ncell = 0;
    DevBuf<float> map_raw;
    DevBuf<unsigned> keys, keys_sorted;
    DevBuf<int> vals, vals_sorted;
    DevBuf<unsigned char> cub_tmp;
    DevBuf<float4> map_pts, map_pts_alt;       // sorted grid points (double-buffered for the incremental merge)
    DevBuf<int> cell_start, cell_start_alt;
    DevBuf<float> map_raw_alt;
    DevBuf<unsigned char> dead, ins;
    DevBuf<int> dead_before, merge_counts, bbox_dev;
    DevBuf<int> vox_unclean, vox_rep, vox_counts;  // Add_Points voxels resolved by the one-thread replay (k_vox_replay*)
    float map_lo[3] = {0, 0, 0}, map_hi[3] = {0, 0, 0};   // tight bounding box of the live map points
    float grid_lo[3] = {0, 0, 0}, grid_hi[3] = {0, 0, 0}; // box the kNN grid covers (= map box + a margin for growth)
    // map maintenance scratch
    DevBuf<float> map_comb, boxes;
    DevBuf<unsigned long long> vkeys, vkeys_sorted;
    DevBuf<unsigned char> keep;
    DevBuf<int> sel_idx;

    // scan + per-point persistent
    int N = 0;
    DevBuf<float> scan_raw;
    DevBuf<unsigned> skeys, skeys_sorted;
    DevBuf<int> svals, svals_sorted;
    DevBuf<float4> scan;
    DevBuf<unsigned char> sel, plane_ok;
    DevBuf<float4> plane;
    // the scan is double-buffered: flb_scan_upload fills the OTHER set on `scan_stream` (copy + ordering kernel) while
    // updates already enqueued on `stream` still read this one, then swaps the two and makes `stream` wait for it
    DevBuf<float4> scan_alt, plane_alt;
    DevBuf<unsigned char> sel_alt, plane_ok_alt;
    cudaStream_t scan_stream = nullptr;
    cudaEvent_t ev_scan_ready = nullptr;
    cudaEvent_t ev_scan_free[2] = {nullptr, nullptr};   // [slot]: everything on `stream` that reads that slot has been enqueued before it
    bool scan_free_valid[2] = {false, false};
    int scan_slot = 0;
    DevBuf<unsigned char> scan_cub_tmp;                 // the upload's own sort scratch (cub_tmp belongs to `stream`)
    int pers_sms = 0;                                   // SMs the persistent kernels may fill (one is left to the scan stream)
    int scan_sort_mode = 0;                             // 0 auto, 1 one-block ordering kernel, 2 device-wide sort (flb_debug_set_scan_sort)
    bool sort_attr_set[3] = {false, false, false};      // dynamic shared memory opt-in of the three k_scan_sort_block instances

    // LIO exports (lazily allocated)
    DevBuf<float> x_world, x_nn_d2, x_pd2, x_pabcd;
    DevBuf<int> x_nn_idx;
    DevBuf<unsigned char> x_rowmask;
    DevBuf<double> x_rows, x_meas;
    int last_pass_width = 0;
    bool last_pass_valid = false;

    // reductions / solve
    DevBuf<double> partials;     // max(nblocks_lio * 92, nblocks_vio * 29)
    DevBuf<double> packed;       // 128
    DevBuf<double> pose12;       // 12
    DevBuf<PriorBlock> prior;    // P11^-1 and P21*P11^-1 of the running update
    DevBuf<double> G_last;       // 108
    DevBuf<State18> states;      // [0]=x [1]=x_prop [2]=old_state(VIO) [3]=saved x [4]=saved x_prop
    DevBuf<StateIkfom> ik_states;   // [0] = x_/P_, [1] = x_propagated/P_propagated
    DevBuf<IkfomCtrl> ik_ctrl;
    int occ_ik = 0;
    DevBuf<LioCtrl> lio_ctrl;
    DevBuf<VioCtrl> vio_ctrl;
    DevBuf<GridBarrier> barrier; // grid barrier of the persistent kernels
    DevBuf<unsigned long long> pkt;    // pose packet of the persistent kernels (kPktUnits flagged words)
    unsigned pkt_epoch = 0;            // flag base of the next launch (flags are never reused, see next_epoch)
    DevBuf<unsigned long long> trace;  // [0..kTraceLen) LIO, [kTraceLen..2*kTraceLen) VIO
    DevBuf<unsigned long long> dbg;    // per-block stage stamps of the last LIO pass (tracing only)
    DevBuf<unsigned long long> dbg_vio;
    DevBuf<double> imu_buf;            // flb_imu_undistort: samples | carry | aux | poses
    DevBuf<float4> imu_pts;            // in | out
    DevBuf<int> imu_heads;
    DevBuf<unsigned long long> vm_key;   // flb_visual_candidates: per-cell {score, ~index}
    DevBuf<float> vm_val, vm_pts;
    DevBuf<int> vm_win;
    DevBuf<double> vm_pose;
    int dbg_vio_blocks = 0;
    int dbg_blocks = 0;
    bool tracing = false;
    int num_sms = 0;
    int occ_lio = 0, occ_vio = 0;
    Staging st_map, st_scan, st_img, st_patch, st_state, st_misc;   // per-kind upload staging
    PinBuf pin_out;              // staging for downloads
    PinBuf pin_res[2];           // flb_state_download_enqueue / _wait: two result slots in flight
    cudaEvent_t ev_res[2] = {nullptr, nullptr};
    bool res_pending[2] = {false, false};
    bool state_valid = false;
    // device-side state moves that the next persistent kernel performs itself instead of a separate D2D copy
    bool reset_pending = false;   // flb_state_reset_enqueue: x, x_prop := the saved pair
    bool prior_pending = false;   // flb_state_set_prior_enqueue: x_prop := x

    // VIO inputs
    int img_w = 0, img_h = 0;
    DevBuf<unsigned char> img, img_alt;
    int Pn = 0;
    DevBuf<double> patch_pos, patch_pos_alt;
    DevBuf<float> patch_ref, patch_ref_alt;
    DevBuf<int> patch_level, patch_level_alt;
    DevBuf<float> errors;        // 2 x err_stride (local shard; the persistent kernel's passes alternate between the halves)
    DevBuf<unsigned long long> err_units;   // 2 x err_stride {tag : error} units (persistent kernel, single GPU: what its leader polls)
    int err_stride = 0;
    DevBuf<float> errors_all;    // padded shard * world (multi-GPU)
    DevBuf<double> x_z, x_H;
    bool cam_set = false;
    CamModel cam{};

    bool last_vio_valid = false;

    // device-resident visual map (rows f2 / f4)
    struct Vm {
        bool on = false;
        VmParams prm{};
        double Rci_Pci[12] = {0};            // camera <- IMU extrinsic (LidarSelector::init, :44-45)
        DevBuf<VmPoint> pts;
        DevBuf<VmFeature> fts;
        DevBuf<unsigned char> pool;          // keyframe images, pool_slots x (w * h)
        int pool_slots = 0;
        int pts_ub = 0, fts_ub = 0, img_ub = 0;   // host-side upper bounds of the device counters
        DevBuf<int> counters;
        DevBuf<double> pose, rci;            // T_f_w of the current frame (12) ; Rci | Pci (12)
        DevBuf<float> pg;                    // scan points of the current call
        DevBuf<unsigned long long> depth, keyset, cell_best, cand_key;
        unsigned key_mask = 0;
        DevBuf<unsigned char> cell_type;
        DevBuf<float> map_value, cell_err, cell_patch, sel_error;
        DevBuf<int> cell_flag, cell_rank, cell_level, cell_point, sel_index, sel_point, winner, scan_tmp;
        Staging st_pg;
    } vm;
    bool pn_on_device = false;   // the patch list was built on the device (flb_vmap_select without a count readback)

    // batched frames (SURVEY.md section 7 H2(iv)): B independent frames per launch, all against the handle's map
    struct Batch {
        int B = 0, n_max = 0, n_cap = 0;
        std::vector<int> N;                  // points per frame
        DevBuf<float4> scan, plane;          // B x n_cap
        DevBuf<unsigned char> sel, plane_ok;
        DevBuf<double> partials;             // B x max(nb_lio * 29, nb_vio * 29)
        size_t partials_per = 0;
        DevBuf<State18> states;              // B x {x, x_prop, old_state, saved x, saved x_prop}
        DevBuf<LioCtrl> lio_ctrl;
        DevBuf<VioCtrl> vio_ctrl;
        DevBuf<PriorBlock> prior;
        DevBuf<double> G_last;               // B x 108
        DevBuf<float> errors;                // B x 2 x err_stride
        DevBuf<LioArgs> lio_args;
        DevBuf<LioSolveArgs> lio_solve;
        DevBuf<VioArgs> vio_args;
        DevBuf<VioSolveArgs> vio_solve;
        DevBuf<LioCtrl*> lio_ctrl_ptrs;
        DevBuf<VioCtrl*> vio_ctrl_ptrs;
    } batch;

    // multi-GPU
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1;
    int err_shard = 0;           // max patches per rank (equal-size ncclAllGather shards)
    // fused NVLink exchange (persistent kernels, no NCCL in the data path)
    DevBuf<P2PMailbox> mailbox;
    DevBuf<unsigned long long> p2p_seq;
    P2PArgs p2p{};               // world <= 1: not attached
    void* p2p_peer_ptr[kP2PMaxWorld] = {nullptr};

    // profiling
    bool profiling = false;
    struct Ev { cudaEvent_t a, b; int fam; };
    std::vector<Ev> evs;
};

namespace {

int fail(flb_handle* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (h) h->err = buf;
    else g_create_error = buf;
    return code;
}

#define FLB_CUDA(h, expr)                                                                         \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            return fail(h, FLB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

#define FLB_CHECK_H(h)                                   \
    do {                                                 \
        if (!(h)) return FLB_ERR_INVALID;                \
        cudaError_t _e = cudaSetDevice((h)->device);     \
        if (_e != cudaSuccess) return fail(h, FLB_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(_e)); \
    } while (0)

// launch bookkeeping: count every kernel; when profiling, bracket it with an event pair
struct LaunchScope {
    flb_handle* h;
    int fam;
    cudaEvent_t a = nullptr, b = nullptr;
    LaunchScope(flb_handle* h_, int fam_) : h(h_), fam(fam_) {
        h->launches++;
        if (h->profiling) {
            cudaEventCreate(&a);
            cudaEventCreate(&b);
            cudaEventRecord(a, h->stream);
        }
    }
    ~LaunchScope() {
        if (h->profiling) {
            cudaEventRecord(b, h->stream);
            h->evs.push_back({a, b, fam});
        }
    }
};
enum { FAM_LIO_KNN = 0, FAM_LIO_PLAIN = 1, FAM_VIO = 2, FAM_SOLVE = 3, FAM_OTHER = 4 };
constexpr int kVioErrCapMax = 40960;     // floats of dynamic shared memory (160 KB) for the VIO leader's error staging

void to_dev_params(const flb_lio_params* p, LioParamsDev& d) {
    std::memcpy(d.R_LI, p->R_LI, sizeof(d.R_LI));
    std::memcpy(d.t_LI, p->t_LI, sizeof(d.t_LI));
    d.sigma = p->laser_point_cov;
    d.max_iteration = p->max_iteration;
    d.conv_rot_deg = p->conv_rot_deg;
    d.conv_pos_cm = p->conv_pos_cm;
}

// LidarSelector::init() constants, src/lidar_selection.cpp:41-52 + set_extrinsic :35-39 (host, once per call)
void to_dev_params(const flb_vio_params* p, VioParamsDev& d) {
    double Rli[9], Pli[3], t[3];
    m3_T(p->R_LI, Rli);
    m3_vec(Rli, p->t_LI, t);
    for (int i = 0; i < 3; ++i) Pli[i] = -t[i];
    m3_mul(p->Rcl, Rli, d.Rci);
    m3_vec(p->Rcl, Pli, t);
    for (int i = 0; i < 3; ++i) d.Pci[i] = t[i] + p->Pcl[i];
    vio_pose_constants(d.Rci, d.Pci, d.Jdphi_dR, d.Jdp_dR);
    d.sigma = p->img_point_cov;
    d.max_iteration = p->max_iteration;
    d.conv_rot_deg = p->conv_rot_deg;
    d.conv_pos_cm = p->conv_pos_cm;
    d.force_all_passes = p->force_all_passes;
    d.single_level = 0;
}

int lio_nblocks(const flb_handle* h) { return (h->N + kLioBlock - 1) / kLioBlock; }
int vio_nblocks(const flb_handle* h) { return (h->Pn + (kVioBlock / 32) - 1) / (kVioBlock / 32); }

int ensure_common(flb_handle* h) {
    FLB_CUDA(h, h->packed.reserve(128));
    FLB_CUDA(h, h->pose12.reserve(12));
    FLB_CUDA(h, h->prior.reserve(1));
    FLB_CUDA(h, h->G_last.reserve(108));
    FLB_CUDA(h, h->states.reserve(5));
    FLB_CUDA(h, h->lio_ctrl.reserve(1));
    FLB_CUDA(h, h->vio_ctrl.reserve(1));
    FLB_CUDA(h, h->barrier.reserve(1));
    FLB_CUDA(h, h->trace.reserve(2 * kTraceLen));
    FLB_CUDA(h, cudaMemset(h->trace.p, 0, 2 * kTraceLen * sizeof(unsigned long long)));
    FLB_CUDA(h, cudaMemset(h->barrier.p, 0, sizeof(GridBarrier)));
    FLB_CUDA(h, h->pkt.reserve(kPktUnits));
    FLB_CUDA(h, cudaMemset(h->pkt.p, 0, kPktUnits * sizeof(unsigned long long)));
    FLB_CUDA(h, cudaMemset(h->lio_ctrl.p, 0, sizeof(LioCtrl)));
    FLB_CUDA(h, cudaMemset(h->vio_ctrl.p, 0, sizeof(VioCtrl)));
    FLB_CUDA(h, cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, h->device));
    {
        // the per-frame persistent kernels fill all SMs but one: the next frame's scan ordering (one block on `scan_stream`)
        // runs there concurrently.  FLB_RESERVE_SM=0 gives that SM back (A/B measurement).
        static const int env_reserve = [] { const char* e = getenv("FLB_RESERVE_SM"); return e ? atoi(e) : 1; }();
        h->pers_sms = (env_reserve && h->num_sms > 2) ? h->num_sms - 1 : h->num_sms;
    }
    FLB_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->occ_lio, k_lio_update_persistent<kLioPersBlock>, kLioPersBlock, 0));
    FLB_CUDA(h, h->ik_states.reserve(2));
    FLB_CUDA(h, h->ik_ctrl.reserve(1));
    FLB_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->occ_ik, k_lio_update_ikfom_persistent<kLioBlock>, kLioBlock, 0));
    // the VIO leader stages the per-patch errors of a pass in dynamic shared memory (up to kVioErrCapMax floats)
    FLB_CUDA(h, cudaFuncSetAttribute(k_vio_update_persistent<kVioPersBlock>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     kVioErrCapMax * (int)sizeof(float)));
    FLB_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->occ_vio, k_vio_update_persistent<kVioPersBlock>, kVioPersBlock,
                                                             kVioErrCapMax * sizeof(float)));
    FLB_CUDA(h, h->pin_out.reserve(1 << 16));
    return FLB_OK;
}

LioArgs make_lio_args(flb_handle* h, const LioParamsDev& prm, bool exports, int width) {
    LioArgs a{};
    a.scan = h->scan.p;
    a.N = h->N;
    a.grid = h->grid;
    a.cell_start = h->cell_start.p;
    a.map_pts = h->map_pts.p;
    a.state = &h->states.p[0];
    a.prm = prm;
    a.plane_thr = (float)h->cfg.plane_threshold;
    a.ctrl = h->lio_ctrl.p;
    a.force_rematch = -1;
    a.pose_override = nullptr;
    a.sel = h->sel.p;
    a.plane = h->plane.p;
    a.plane_ok = h->plane_ok.p;
    a.partials = h->partials.p;
    a.M = h->M;
    a.prefetch = 0;
    if (exports) {
        a.x_world = h->x_world.p;
        a.x_nn_idx = h->x_nn_idx.p;
        a.x_nn_d2 = h->x_nn_d2.p;
        a.x_pabcd = h->x_pabcd.p;
        a.x_pd2 = h->x_pd2.p;
        a.x_rowmask = h->x_rowmask.p;
        a.x_rows = h->x_rows.p;
        a.x_meas = h->x_meas.p;
    }
    (void)width;
    return a;
}

int launch_lio_pass(flb_handle* h, const LioArgs& a, int width, bool knn_family) {
    const int nb = lio_nblocks(h);
    if (nb == 0) return FLB_OK;
    LaunchScope ls(h, knn_family ? FAM_LIO_KNN : FAM_LIO_PLAIN);
    if (width == 6) k_lio_pass<6, kLioBlock><<<nb, kLioBlock, 0, h->stream>>>(a);
    else k_lio_pass<12, kLioBlock><<<nb, kLioBlock, 0, h->stream>>>(a);
    FLB_CUDA(h, cudaGetLastError());
    return FLB_OK;
}

// all-reduce of the packed sums (and all-gather of the per-patch errors) for multi-GPU
int allreduce_packed(flb_handle* h, const double* partials, int nblocks, int K) {
    {
        LaunchScope ls(h, FAM_SOLVE);
        k_reduce_only<<<1, 32, 0, h->stream>>>(partials, nblocks, K, h->packed.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    int r = g_nccl.AllReduce(h->packed.p, h->packed.p, (size_t)K, kNcclFloat64, kNcclSum, h->comm, h->stream);
    if (r != 0) return fail(h, FLB_ERR_COMM, "ncclAllReduce: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
    h->launches++;
    return FLB_OK;
}

// true when p is page-locked host memory (flb_host_alloc / cudaHostAlloc / cudaHostRegister): the copy engine
// can read it directly, so the staging memcpy is skipped
bool is_pinned(const void* p) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// copy_stream is about to fill the OTHER set of a double-buffered input.  Every reader of the current set has been
// enqueued on `stream` by now (record its event); the other set's readers were all enqueued before the previous upload,
// whose event the copy waits for.
int vio_copy_begin(flb_handle* h, flb_handle::InSlot& s) {
    for (int k = 0; k < 2; ++k)
        if (!s.free_ev[k]) FLB_CUDA(h, cudaEventCreateWithFlags(&s.free_ev[k], cudaEventDisableTiming));
    FLB_CUDA(h, cudaEventRecord(s.free_ev[s.slot], h->stream));
    s.valid[s.slot] = true;
    if (s.valid[s.slot ^ 1]) FLB_CUDA(h, cudaStreamWaitEvent(h->copy_stream, s.free_ev[s.slot ^ 1], 0));
    return FLB_OK;
}
int vio_copy_end(flb_handle* h) {
    FLB_CUDA(h, cudaEventRecord(h->ev_vio_inputs, h->copy_stream));
    h->vio_inputs_pending = true;
    return FLB_OK;
}
// a kernel on `stream` is about to read the image / patches
int vio_inputs_acquire(flb_handle* h) {
    if (h->vio_inputs_pending) {
        FLB_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_vio_inputs, 0));
        h->vio_inputs_pending = false;
    }
    return FLB_OK;
}
int vio_inputs_release(flb_handle*) { return FLB_OK; }   // (readers are fenced per slot at the next upload: vio_copy_begin)

// Perform the deferred device-side state moves with plain copies (every consumer other than the persistent kernels).
int flush_state_ops(flb_handle* h) {
    if (h->reset_pending) {
        FLB_CUDA(h, cudaMemcpyAsync(&h->states.p[0], &h->states.p[3], 2 * sizeof(State18), cudaMemcpyDeviceToDevice, h->stream));
        h->reset_pending = false;
    }
    if (h->prior_pending) {
        FLB_CUDA(h, cudaMemcpyAsync(&h->states.p[1], &h->states.p[0], sizeof(State18), cudaMemcpyDeviceToDevice, h->stream));
        h->prior_pending = false;
    }
    return FLB_OK;
}

// Flag base for one persistent launch: flags epoch+1 .. epoch+4095 belong to it alone.  On wrap-around the
// packet is cleared (stream-ordered) so that no stale unit can ever match.
int next_epoch(flb_handle* h, unsigned* epoch) {
    if (h->pkt_epoch >= 0xFFFF0000u || h->pkt_epoch == 0) {
        if (h->pkt_epoch) FLB_CUDA(h, cudaMemsetAsync(h->pkt.p, 0, kPktUnits * sizeof(unsigned long long), h->stream));
        h->pkt_epoch = 4096;
    }
    *epoch = h->pkt_epoch;
    h->pkt_epoch += 4096;
    return FLB_OK;
}

int enqueue_lio_update(flb_handle* h, const flb_lio_params* prm) {
    // fused multi-GPU mode: a rank whose shard is empty still launches (its leader takes part in every exchange)
    if (h->M <= 0 || (h->N <= 0 && !(h->p2p.world > 1 && h->scan.p)))
        return fail(h, FLB_ERR_STATE, "flb_lio_update: map and scan must be uploaded first");
    if (!h->state_valid) return fail(h, FLB_ERR_STATE, "flb_lio_update: no device state (flb_state_upload)");
    if (prm->max_iteration < 0 || prm->max_iteration > 1000) return fail(h, FLB_ERR_INVALID, "max_iteration outside [0, 1000]");
    if (h->p2p.world > 1 && !h->cfg.persistent)
        return fail(h, FLB_ERR_STATE, "the fused NVLink exchange lives in the persistent kernels (flb_config.persistent = 1)");
    LioParamsDev d;
    to_dev_params(prm, d);
    LioSolveArgs s{};
    s.state = &h->states.p[0];
    s.state_prop = &h->states.p[1];
    s.ctrl = h->lio_ctrl.p;
    s.prior = h->prior.p;
    s.partials = h->partials.p;
    s.nblocks = lio_nblocks(h);
    s.prm = d;
    s.p2p = h->p2p;
    s.timeout_flag = &h->barrier.p->timeout;
    LioArgs a = make_lio_args(h, d, false, 6);
    const bool lio_persistent = h->cfg.persistent && (!h->comm || h->p2p.world > 1);
    if (h->prior_pending || (h->reset_pending && !lio_persistent)) { int rcf = flush_state_ops(h); if (rcf) return rcf; }
    if (h->reset_pending) {              // the kernel starts from the saved pair and restores state / state_prop itself
        s.init_x = &h->states.p[3];
        s.init_xp = &h->states.p[4];
        h->reset_pending = false;
    }
    if (lio_persistent) {
        // one cooperative launch for the whole iterated update; grid = min(needed, co-resident capacity)
        // whole multiples of the SM count (<= co-resident capacity): chunks are dealt round-robin to blocks
        // worker blocks (one per SM, chunks dealt round-robin) + one leader block
        const int cap = std::min(h->occ_lio * h->num_sms, h->pers_sms);
        if (cap < 2) return fail(h, FLB_ERR_STATE, "persistent mode needs two co-resident blocks");
        const int workers = std::max(1, std::min((h->N + 31) / 32, cap - 1));
        const int grid = workers + 1;
        FLB_CUDA(h, h->partials.reserve(std::max<size_t>((size_t)grid * lio_packed(12), h->partials.cap)));
        a.partials = h->partials.p;
        s.partials = h->partials.p;
        s.nblocks = workers;
        GridBarrier* bar = h->barrier.p;
        unsigned long long* trace = h->tracing ? h->trace.p : nullptr;
        a.probe = h->tracing ? h->trace.p + 112 : nullptr;
        a.chunk = std::max(1, std::min(32, (h->N + workers * (kLioPersBlock / 32) - 1) / (workers * (kLioPersBlock / 32))));
        {
            static const int env_warm = [] { const char* e = getenv("FLB_WARM"); return e ? atoi(e) : 1; }();
            if (env_warm) {
                WarmList& w = a.warm;
                const size_t n1 = (size_t)std::max(h->N, 1);
                const void* ptr[] = {h->scan.p, h->map_pts.p, h->cell_start.p, h->plane.p, h->sel.p, h->plane_ok.p, h->partials.p, h->states.p};
                const size_t len[] = {n1 * 16, (size_t)h->M * 16, ((size_t)h->ncell + 1) * 4, n1 * 16, n1, n1, (size_t)grid * lio_packed(6) * 8,
                                      5 * sizeof(State18)};
                w.n = 8;
                for (int k = 0; k < 8; ++k) { w.p[k] = ptr[k]; w.bytes[k] = len[k]; }
            }
        }
        {
            // L2 prefetch of the map (points + cell table) at kernel start: on by default (C2, 5.3 MB: first pass 36.1 -> 34.0 us,
            // +1.2 % frames/s; C3, 27 MB: 250 -> 239 us); FLB_PREFETCH=0/1 overrides
            const size_t bytes = (size_t)h->M * 16 + ((size_t)h->ncell + 1) * 4;
            static const int env = [] { const char* e = getenv("FLB_PREFETCH"); return e ? atoi(e) : -1; }();
            a.prefetch = env >= 0 ? env : (bytes > (1u << 20) ? 1 : 0);
        }
        unsigned long long* dbg = nullptr;
        if (h->tracing) {
            FLB_CUDA(h, h->dbg.reserve((size_t)grid * 16));
            FLB_CUDA(h, cudaMemsetAsync(h->dbg.p, 0, (size_t)grid * 16 * sizeof(unsigned long long), h->stream));
            h->dbg_blocks = grid;
            dbg = h->dbg.p;
        }
        unsigned long long* pkt = h->pkt.p;
        unsigned epoch = 0;
        { int rce = next_epoch(h, &epoch); if (rce) return rce; }
        void* args[] = {&a, &s, &bar, &pkt, &epoch, &trace, &dbg};
        LaunchScope ls(h, FAM_LIO_KNN);
        FLB_CUDA(h, cudaLaunchCooperativeKernel((void*)k_lio_update_persistent<kLioPersBlock>, dim3(grid), dim3(kLioPersBlock), args, 0,
                                                h->stream));
        h->last_pass_valid = false;
        return FLB_OK;
    }
    {
        LaunchScope ls(h, FAM_SOLVE);
        k_lio_begin<<<1, 32, 0, h->stream>>>(h->lio_ctrl.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    const int T = prm->max_iteration;
    for (int it = -1; it < T; ++it) {
        // Statically known rematch schedule when early stop is disabled is NOT assumed here:
        // the kernel reads ctrl->nearest_search_en / ctrl->stop on the device.
        int rc = launch_lio_pass(h, a, 6, it == -1);
        if (rc) return rc;
        if (h->comm) {
            rc = allreduce_packed(h, h->partials.p, lio_nblocks(h), lio_packed(6));
            if (rc) return rc;
            s.partials = h->packed.p;
            s.nblocks = 1;
        }
        LaunchScope ls(h, FAM_SOLVE);
        k_lio_finalize<<<1, kLeaderBlock, 0, h->stream>>>(s);
        FLB_CUDA(h, cudaGetLastError());
    }
    h->last_pass_valid = false;
    return FLB_OK;
}

// The patch list of the last flb_vmap_select lives on the device; calls that need its length on the host fetch it here.
int resolve_pn(flb_handle* h) {
    if (!h->pn_on_device) return FLB_OK;
    int n = 0;
    FLB_CUDA(h, cudaMemcpyAsync(&n, h->vm.counters.p + VM_N_SEL, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    h->Pn = n;
    h->pn_on_device = false;
    return FLB_OK;
}

int enqueue_vio_update(flb_handle* h, const flb_vio_params* prm) {
    if (!h->cam_set || h->img_w <= 0) return fail(h, FLB_ERR_STATE, "flb_vio_update: camera and image must be set first");
    if (h->cam.width != h->img_w || h->cam.height != h->img_h) return fail(h, FLB_ERR_STATE, "camera / image size mismatch");
    if (!h->state_valid) return fail(h, FLB_ERR_STATE, "flb_vio_update: no device state (flb_state_upload)");
    if (prm->max_iteration > 1000) return fail(h, FLB_ERR_INVALID, "max_iteration outside [0, 1000]");
    if (h->pn_on_device && !(h->cfg.persistent && h->p2p.world <= 1 && !h->comm && prm->max_iteration > 0)) {
        int rcp = resolve_pn(h);             // only the single-GPU persistent kernel reads the count on the device
        if (rcp) return rcp;
    }
    VioParamsDev d;
    to_dev_params(prm, d);
    VioSolveArgs s{};
    s.state = &h->states.p[0];
    s.state_prop = &h->states.p[1];
    s.old_state = &h->states.p[2];
    s.ctrl = h->vio_ctrl.p;
    s.prior = h->prior.p;
    s.G_last = h->G_last.p;
    s.partials = h->partials.p;
    s.nblocks = vio_nblocks(h);
    s.errors = h->errors.p;
    s.err_stride = h->err_stride;
    s.Pn_total = h->Pn;
    s.prm = d;
    s.p2p = h->p2p;
    s.timeout_flag = &h->barrier.p->timeout;
    { int rcq = vio_inputs_acquire(h); if (rcq) return rcq; }
    const bool fused = h->p2p.world > 1;
    if (fused && !h->cfg.persistent)
        return fail(h, FLB_ERR_STATE, "the fused NVLink exchange lives in the persistent kernels (flb_config.persistent = 1)");
    if (fused && h->Pn > kP2PErrCap) return fail(h, FLB_ERR_INVALID, "fused multi-GPU mode: at most %d patches per rank", kP2PErrCap);
    const bool persistent = h->cfg.persistent && (fused || (!h->comm && (h->Pn > 0 || h->pn_on_device))) && prm->max_iteration > 0;
    if (h->reset_pending || (h->prior_pending && !persistent)) { int rcf = flush_state_ops(h); if (rcf) return rcf; }
    if (h->prior_pending) {              // the kernel takes state_propagat = state itself
        s.prior_from_state = 1;
        h->prior_pending = false;
    }
    if (!persistent) {
        LaunchScope ls(h, FAM_SOLVE);
        k_vio_begin<<<1, 32, 0, h->stream>>>(h->vio_ctrl.p, h->Pn);
        FLB_CUDA(h, cudaGetLastError());
    }
    VioArgs a{};
    a.img = h->img.p;
    a.cam = h->cam;
    a.pos = h->patch_pos.p;
    a.patch = h->patch_ref.p;
    a.search_level = h->patch_level.p;
    a.Pn = h->Pn;
    a.state = &h->states.p[0];
    a.pose_override = nullptr;
    a.prm = d;
    a.ctrl = h->vio_ctrl.p;
    a.force_level = -1;
    a.errors = h->errors.p;
    a.err_stride = h->err_stride;
    a.partials = h->partials.p;
    a.p2p = h->p2p;
    a.Pn_dev = nullptr;
    if (h->pn_on_device) {                   // capacity = one patch per grid cell; the kernel reads the real count
        a.Pn = h->vm.prm.length;
        a.Pn_dev = h->vm.counters.p + VM_N_SEL;
        s.Pn_total = a.Pn;
    }
    const int nb = vio_nblocks(h);
    static const int env_defer = [] { const char* e = getenv("FLB_DEFER"); return e ? atoi(e) : 1; }();
    if (persistent && !fused && env_defer) {
        // per-patch errors as self-validating units (zeroed once per allocation: a tag always has its top bit set)
        const size_t need = 2 * (size_t)std::max(h->err_stride, 1);
        if (need > h->err_units.cap) {
            FLB_CUDA(h, h->err_units.reserve(need));
            FLB_CUDA(h, cudaMemsetAsync(h->err_units.p, 0, h->err_units.cap * sizeof(unsigned long long), h->stream));
        }
        a.err_units = h->err_units.p;
        s.err_units = h->err_units.p;
    }
    if (persistent) {
        // patches are dealt warp-round-robin over the worker blocks; one more block is the leader
        const int cap = std::min(h->occ_vio * h->num_sms, h->pers_sms);
        if (cap < 2) return fail(h, FLB_ERR_STATE, "persistent mode needs two co-resident blocks");
        const int workers = std::max(1, std::min(std::max(a.Pn, 1), cap - 1));
        const int grid = workers + 1;
        FLB_CUDA(h, h->partials.reserve(std::max<size_t>((size_t)grid * kVioPacked, h->partials.cap)));
        a.partials = h->partials.p;
        s.partials = h->partials.p;
        s.nblocks = workers;
        GridBarrier* bar = h->barrier.p;
        unsigned long long* trace = h->tracing ? h->trace.p + kTraceLen : nullptr;
        unsigned long long* pkt = h->pkt.p;
        unsigned epoch = 0;
        { int rce = next_epoch(h, &epoch); if (rce) return rce; }
        unsigned long long* dbg = nullptr;
        if (h->tracing) {
            FLB_CUDA(h, h->dbg_vio.reserve((size_t)grid * kVioDbg));
            FLB_CUDA(h, cudaMemsetAsync(h->dbg_vio.p, 0, (size_t)grid * kVioDbg * sizeof(unsigned long long), h->stream));
            dbg = h->dbg_vio.p;
            h->dbg_vio_blocks = grid;
        }
        // staging capacity for the errors of ALL ranks (the peers' shard sizes are not known here: assume like ours + slack)
        int err_cap = (int)std::min<long long>(kVioErrCapMax, std::max<long long>(2048, ((long long)a.Pn * std::max(h->p2p.world, 1) * 5 / 4 + 319) / 256 * 256));
        {
            static const int env_warm = [] { const char* e = getenv("FLB_WARM"); return e ? atoi(e) : 1; }();
            if (env_warm) {
                WarmList& w = a.warm;
                const size_t pn = (size_t)std::max(a.Pn, 1);
                const void* ptr[] = {h->img.p, h->patch_pos.p, h->patch_ref.p, h->patch_level.p, h->errors.p, h->partials.p};
                const size_t len[] = {(size_t)h->img_w * h->img_h, pn * 24, pn * 768, pn * 4, 2 * (size_t)h->err_stride * 4, (size_t)grid * kVioPacked * 8};
                w.n = 6;
                for (int k = 0; k < 6; ++k) { w.p[k] = ptr[k]; w.bytes[k] = len[k]; }
            }
        }
        const size_t dyn = (size_t)err_cap * sizeof(float);
        void* args[] = {&a, &s, &bar, &pkt, &epoch, &trace, &dbg, &err_cap};
        LaunchScope ls(h, FAM_VIO);
        FLB_CUDA(h, cudaLaunchCooperativeKernel((void*)k_vio_update_persistent<kVioPersBlock>, dim3(grid), dim3(kVioPersBlock), args, dyn,
                                                h->stream));
        h->last_vio_valid = false;
        return vio_inputs_release(h);
    }
    const int total = 3 * std::max(prm->max_iteration, 0);
    for (int it = 0; it < total && h->Pn > 0; ++it) {
        {
            LaunchScope ls(h, FAM_VIO);
            k_vio_pass<kVioBlock><<<nb, kVioBlock, 0, h->stream>>>(a);
            FLB_CUDA(h, cudaGetLastError());
        }
        if (h->comm) {
            int rc = allreduce_packed(h, h->partials.p, nb, kVioPacked);
            if (rc) return rc;
            s.partials = h->packed.p;
            s.nblocks = 1;
            // gather every rank's per-patch errors in patch order (shards padded to errors.cap/world)
            const size_t shard = (size_t)h->err_shard;
            int r = g_nccl.AllGather(h->errors.p, h->errors_all.p, shard, kNcclFloat32, h->comm, h->stream);
            if (r != 0) return fail(h, FLB_ERR_COMM, "ncclAllGather failed");
            h->launches++;
            s.errors = h->errors_all.p;
            s.Pn_total = (int)(shard * (size_t)h->world);
        }
        LaunchScope ls(h, FAM_SOLVE);
        k_vio_finalize<<<1, kLeaderBlock, 0, h->stream>>>(s);
        FLB_CUDA(h, cudaGetLastError());
    }
    h->last_vio_valid = false;
    return vio_inputs_release(h);
}

void fill_lio_report(const LioCtrl& c, flb_lio_report* rep) {
    rep->passes = c.passes;
    rep->knn_passes = c.knn_passes;
    rep->n_eff_last = c.n_eff_last;
    rep->res_mean_last = c.res_mean_last;
    rep->rows_total = c.rows_total;
    rep->converged_last = c.converged_last;
    rep->status = c.status;
}
void fill_vio_report(const VioCtrl& c, flb_vio_report* rep) {
    for (int l = 0; l < 3; ++l) { rep->passes[l] = c.passes[l]; rep->last_error[l] = c.level_error[l]; }
    rep->rows_total = c.rows_total;
    rep->skipped_last = c.skipped_last;
    rep->cov_updated = c.cov_updated;
    rep->status = c.status;
}

}  // namespace

template <int kScanSortBlock, int ITEMS>
static int launch_scan_sort_block(flb_handle* h, cudaStream_t ss, int N, const float lo[3], float inv_cell) {
    using Sort = cub::BlockRadixSort<unsigned, kScanSortBlock, ITEMS, int, 6>;
    const size_t smem = std::max(sizeof(typename Sort::TempStorage), (size_t)kScanSortBlock * ITEMS * sizeof(unsigned));
    bool& attr_set = h->sort_attr_set[ITEMS == 17 ? 0 : (ITEMS == 33 ? 1 : 2)];      // per handle: the attribute is per device
    if (!attr_set) {
        FLB_CUDA(h, cudaFuncSetAttribute(k_scan_sort_block<kScanSortBlock, ITEMS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    k_scan_sort_block<kScanSortBlock, ITEMS><<<1, kScanSortBlock, smem, ss>>>(h->scan_raw.p, N, lo[0], lo[1], lo[2], inv_cell, h->scan_alt.p, h->sel_alt.p,
                                                             h->plane_ok_alt.p);
    FLB_CUDA(h, cudaGetLastError());
    return FLB_OK;
}

extern "C" {

int flb_abi_version(void) { return FLB_ABI_VERSION; }

const char* flb_last_error(const flb_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int flb_create(const flb_config* cfg, flb_handle** out) {
    if (!out) return FLB_ERR_INVALID;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, FLB_ERR_NO_DEVICE,
                    "no CUDA device (%s): fastlivo_b200 has no CPU fallback", e == cudaSuccess ? "count = 0" : cudaGetErrorString(e));
    flb_config c{};
    c.persistent = 1;
    if (cfg) c = *cfg;
    if (c.device < 0 || c.device >= ndev) return fail(nullptr, FLB_ERR_INVALID, "device %d out of range [0,%d)", c.device, ndev);
    if (!(c.cell_size > 0)) c.cell_size = 0.6;
    if (!(c.knn_max_d2 > 0)) c.knn_max_d2 = 5.0;
    if (!(c.plane_threshold > 0)) c.plane_threshold = 0.1;
    e = cudaSetDevice(c.device);
    if (e != cudaSuccess) return fail(nullptr, FLB_ERR_CUDA, "cudaSetDevice(%d): %s", c.device, cudaGetErrorString(e));
    flb_handle* h = new flb_handle;
    h->device = c.device;
    h->cfg = c;
    e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete h;
        return fail(nullptr, FLB_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    }
    h->stream = h->own_stream;
    if (cudaStreamCreateWithFlags(&h->scan_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_scan_ready, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_scan_free[0], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_scan_free[1], cudaEventDisableTiming) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_vio_inputs, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_vio_done, cudaEventDisableTiming) != cudaSuccess) {
        cudaStreamDestroy(h->own_stream);
        delete h;
        return fail(nullptr, FLB_ERR_CUDA, "copy stream / event creation failed");
    }
    int rc = ensure_common(h);
    if (rc) {
        g_create_error = h->err;
        cudaStreamDestroy(h->own_stream);
        delete h;
        return rc;
    }
    *out = h;
    return FLB_OK;
}

int flb_destroy(flb_handle* h) {
    if (!h) return FLB_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    for (int r = 0; r < kP2PMaxWorld; ++r)
        if (h->p2p_peer_ptr[r]) cudaIpcCloseMemHandle(h->p2p_peer_ptr[r]);
    h->mailbox.release();
    h->p2p_seq.release();
    {
        auto& b = h->batch;
        b.scan.release(); b.plane.release(); b.sel.release(); b.plane_ok.release(); b.partials.release(); b.states.release();
        b.lio_ctrl.release(); b.vio_ctrl.release(); b.prior.release(); b.G_last.release(); b.errors.release(); b.lio_args.release();
        b.lio_solve.release(); b.vio_args.release(); b.vio_solve.release(); b.lio_ctrl_ptrs.release(); b.vio_ctrl_ptrs.release();
    }
    {
        auto& vm = h->vm;
        vm.pts.release(); vm.fts.release(); vm.pool.release(); vm.counters.release(); vm.pose.release(); vm.rci.release(); vm.pg.release();
        vm.depth.release(); vm.keyset.release(); vm.cell_best.release(); vm.cand_key.release(); vm.cell_type.release(); vm.map_value.release();
        vm.cell_err.release(); vm.cell_patch.release(); vm.sel_error.release(); vm.cell_flag.release(); vm.cell_rank.release();
        vm.cell_level.release(); vm.cell_point.release(); vm.sel_index.release(); vm.sel_point.release(); vm.winner.release();
        vm.scan_tmp.release(); vm.st_pg.release();
    }
    for (auto& ev : h->evs) { cudaEventDestroy(ev.a); cudaEventDestroy(ev.b); }
    h->map_raw.release(); h->keys.release(); h->keys_sorted.release(); h->vals.release(); h->vals_sorted.release();
    h->map_comb.release(); h->boxes.release(); h->vkeys.release(); h->vkeys_sorted.release(); h->keep.release(); h->sel_idx.release();
    h->map_pts_alt.release(); h->cell_start_alt.release(); h->map_raw_alt.release(); h->dead.release(); h->ins.release();
    h->dead_before.release(); h->merge_counts.release(); h->bbox_dev.release();
    h->vox_unclean.release(); h->vox_rep.release(); h->vox_counts.release();
    h->cub_tmp.release(); h->map_pts.release(); h->cell_start.release(); h->scan.release(); h->sel.release();
    h->plane_ok.release(); h->plane.release(); h->x_world.release(); h->x_nn_d2.release(); h->x_pd2.release();
    h->x_nn_idx.release(); h->x_rowmask.release(); h->x_rows.release(); h->x_meas.release(); h->partials.release();
    h->packed.release(); h->pose12.release(); h->prior.release(); h->scan_raw.release(); h->skeys.release(); h->skeys_sorted.release(); h->svals.release(); h->svals_sorted.release(); h->x_pabcd.release(); h->G_last.release(); h->states.release();
    h->lio_ctrl.release(); h->vio_ctrl.release(); h->ik_states.release(); h->ik_ctrl.release(); h->barrier.release(); h->pkt.release(); h->trace.release(); h->dbg.release(); h->dbg_vio.release(); h->imu_buf.release(); h->imu_pts.release(); h->imu_heads.release(); h->vm_key.release(); h->vm_val.release(); h->vm_pts.release(); h->vm_win.release(); h->vm_pose.release(); h->img.release(); h->patch_pos.release(); h->patch_ref.release();
    h->patch_level.release(); h->errors.release(); h->err_units.release(); h->errors_all.release(); h->x_z.release(); h->x_H.release();
    h->st_map.release(); h->st_scan.release(); h->st_img.release(); h->st_patch.release(); h->st_state.release();
    h->st_misc.release(); h->pin_out.release();
    for (int k = 0; k < 2; ++k) { h->pin_res[k].release(); if (h->ev_res[k]) cudaEventDestroy(h->ev_res[k]); }
    cudaStreamSynchronize(h->copy_stream);
    cudaStreamSynchronize(h->scan_stream);
    h->scan_alt.release(); h->plane_alt.release(); h->sel_alt.release(); h->plane_ok_alt.release();
    h->img_alt.release(); h->patch_pos_alt.release(); h->patch_ref_alt.release(); h->patch_level_alt.release();
    for (int k = 0; k < 2; ++k) {
        if (h->img_slot.free_ev[k]) cudaEventDestroy(h->img_slot.free_ev[k]);
        if (h->patch_slot.free_ev[k]) cudaEventDestroy(h->patch_slot.free_ev[k]);
    }
    cudaEventDestroy(h->ev_scan_ready);
    cudaEventDestroy(h->ev_scan_free[0]);
    cudaEventDestroy(h->ev_scan_free[1]);
    h->scan_cub_tmp.release();
    cudaStreamDestroy(h->scan_stream);
    cudaEventDestroy(h->ev_vio_inputs);
    cudaEventDestroy(h->ev_vio_done);
    cudaStreamDestroy(h->copy_stream);
    cudaStreamDestroy(h->own_stream);
    delete h;
    return FLB_OK;
}

int flb_set_stream(flb_handle* h, void* cuda_stream) {
    FLB_CHECK_H(h);
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    return FLB_OK;
}

int flb_synchronize(flb_handle* h) {
    FLB_CHECK_H(h);
    FLB_CUDA(h, cudaStreamSynchronize(h->copy_stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->scan_stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    return FLB_OK;
}

int flb_host_alloc(flb_handle* h, size_t bytes, void** out) {
    FLB_CHECK_H(h);
    if (!out || bytes == 0) return fail(h, FLB_ERR_INVALID, "flb_host_alloc: bad arguments");
    FLB_CUDA(h, cudaHostAlloc(out, bytes, cudaHostAllocDefault));
    return FLB_OK;
}

int flb_host_free(flb_handle* h, void* p) {
    FLB_CHECK_H(h);
    if (p) FLB_CUDA(h, cudaFreeHost(p));
    return FLB_OK;
}

int64_t flb_launch_count(const flb_handle* h) { return h ? h->launches : 0; }

// ---------------------------------------------------------------------------------------
// Build the sorted uniform kNN grid over h->map_raw[0..M) with the bounding box h->map_lo/hi.
static int rebuild_grid(flb_handle* h, int M) {
    // the grid covers the map box plus a margin, so that points added next to the map (a moving sensor) fall inside
    // it and take the incremental path of flb_map_add_points; kNN is exact for any cell geometry
    for (int k = 0; k < 3; ++k) {
        // a whole number of cells, so that the cell boundaries stay where a grid anchored at the map's own corner puts them
        const float cs = (float)h->cfg.cell_size;
        const float m = cs * std::ceil(std::max(2.0f * cs, 0.05f * (h->map_hi[k] - h->map_lo[k])) / cs);
        h->grid_lo[k] = h->map_lo[k] - m;
        h->grid_hi[k] = h->map_hi[k] + m;
    }
    const float* lo = h->grid_lo;
    const float* hi = h->grid_hi;
    // grid geometry; enlarge the cell if the dense grid would exceed 2^25 cells (still exact, just slower)
    double cell = h->cfg.cell_size;
    for (;;) {
        const double nx = std::floor((hi[0] - lo[0]) / cell) + 1, ny = std::floor((hi[1] - lo[1]) / cell) + 1,
                     nz = std::floor((hi[2] - lo[2]) / cell) + 1;
        if (nx * ny * nz <= (double)(1 << 25)) break;
        cell *= 1.26;
    }
    GridDesc g{};
    g.ox = lo[0]; g.oy = lo[1]; g.oz = lo[2];
    g.cell = (float)cell;
    g.inv_cell = 1.0f / g.cell;
    g.nx = (int)std::floor((hi[0] - lo[0]) / cell) + 1;
    g.ny = (int)std::floor((hi[1] - lo[1]) / cell) + 1;
    g.nz = (int)std::floor((hi[2] - lo[2]) / cell) + 1;
    g.max_d2 = (float)h->cfg.knn_max_d2;
    g.max_ring = (int)std::ceil(std::sqrt(h->cfg.knn_max_d2) / cell) + 1;
    const int ncell = g.nx * g.ny * g.nz;
    FLB_CUDA(h, h->keys.reserve(M));
    FLB_CUDA(h, h->keys_sorted.reserve(M));
    FLB_CUDA(h, h->vals.reserve(M));
    FLB_CUDA(h, h->vals_sorted.reserve(M));
    FLB_CUDA(h, h->map_pts.reserve(M));
    FLB_CUDA(h, h->cell_start.reserve((size_t)ncell + 1));
    const int nb = (M + 255) / 256;
    {
        LaunchScope ls(h, FAM_OTHER);
        k_map_cell_ids<<<nb, 256, 0, h->stream>>>(h->map_raw.p, M, 3, g, h->keys.p, h->vals.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    int end_bit = 1;
    while ((1u << end_bit) < (unsigned)ncell && end_bit < 32) ++end_bit;
    size_t tmp_bytes = 0;
    FLB_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, h->keys.p, h->keys_sorted.p, h->vals.p, h->vals_sorted.p, M,
                                                0, end_bit, h->stream));
    FLB_CUDA(h, h->cub_tmp.reserve(tmp_bytes));
    FLB_CUDA(h, cub::DeviceRadixSort::SortPairs(h->cub_tmp.p, tmp_bytes, h->keys.p, h->keys_sorted.p, h->vals.p,
                                                h->vals_sorted.p, M, 0, end_bit, h->stream));
    h->launches += 4;
    {
        LaunchScope ls(h, FAM_OTHER);
        k_map_gather<<<nb, 256, 0, h->stream>>>(h->map_raw.p, M, 3, h->vals_sorted.p, h->map_pts.p);
        k_cell_starts<<<(ncell + 256) / 256, 256, 0, h->stream>>>(h->keys_sorted.p, M, h->cell_start.p, ncell);
        FLB_CUDA(h, cudaGetLastError());
        h->launches++;
    }
    h->M = M;
    h->grid = g;
    h->ncell = ncell;
    return FLB_OK;
}

int flb_map_upload(flb_handle* h, const float* xyz, int M, int stride) {
    FLB_CHECK_H(h);
    if (!xyz || M < 1 || stride < 3) return fail(h, FLB_ERR_INVALID, "flb_map_upload: bad arguments (M=%d stride=%d)", M, stride);
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    void* stv = nullptr;
    FLB_CUDA(h, h->st_map.acquire((size_t)M * 3 * sizeof(float), &stv));
    float* st = static_cast<float*>(stv);
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = 0; i < M; ++i) {
        for (int k = 0; k < 3; ++k) {
            const float v = xyz[(size_t)i * stride + k];
            if (!std::isfinite(v)) return fail(h, FLB_ERR_INVALID, "flb_map_upload: non-finite coordinate at point %d", i);
            st[3 * (size_t)i + k] = v;
            lo[k] = std::min(lo[k], v);
            hi[k] = std::max(hi[k], v);
        }
    }
    for (int k = 0; k < 3; ++k) { h->map_lo[k] = lo[k]; h->map_hi[k] = hi[k]; }
    FLB_CUDA(h, h->map_raw.reserve((size_t)M * 3));
    FLB_CUDA(h, cudaMemcpyAsync(h->map_raw.p, st, (size_t)M * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    int rc = rebuild_grid(h, M);
    if (rc) return rc;
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    return FLB_OK;
}

// ---- device-resident map maintenance (SURVEY.md section 8 row f1) -----------------------------------
// Compact h->map_comb by h->keep flags (positions given by idx_in) into map_raw, then rebuild the grid.
static int compact_and_rebuild(flb_handle* h, const int* idx_in, int total) {
    FLB_CUDA(h, h->sel_idx.reserve((size_t)total + 1));
    size_t tmp_bytes = 0;
    int* d_count = h->sel_idx.p + total;
    FLB_CUDA(h, cub::DeviceSelect::Flagged(nullptr, tmp_bytes, idx_in, h->keep.p, h->sel_idx.p, d_count, total, h->stream));
    FLB_CUDA(h, h->cub_tmp.reserve(tmp_bytes));
    FLB_CUDA(h, cub::DeviceSelect::Flagged(h->cub_tmp.p, tmp_bytes, idx_in, h->keep.p, h->sel_idx.p, d_count, total, h->stream));
    h->launches += 2;
    int count = 0;
    FLB_CUDA(h, cudaMemcpyAsync(&count, d_count, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    if (count < 1) return fail(h, FLB_ERR_STATE, "map maintenance would leave an empty map");
    FLB_CUDA(h, h->map_raw.reserve((size_t)count * 3));   // never shrinks; grows only if count > capacity
    FLB_CUDA(h, h->bbox_dev.reserve(6));
    const int init[6] = {0x7fffffff, 0x7fffffff, 0x7fffffff, (int)0x80000000, (int)0x80000000, (int)0x80000000};
    FLB_CUDA(h, cudaMemcpyAsync(h->bbox_dev.p, init, sizeof(init), cudaMemcpyHostToDevice, h->stream));
    {
        LaunchScope ls(h, FAM_OTHER);
        k_gather_xyz<<<(count + 255) / 256, 256, 0, h->stream>>>(h->map_comb.p, h->sel_idx.p, count, h->map_raw.p);
        k_bbox<<<std::min((count + 255) / 256, 4 * std::max(h->num_sms, 1)), 256, 0, h->stream>>>(h->map_raw.p, count, h->bbox_dev.p);
        FLB_CUDA(h, cudaGetLastError());
        h->launches++;
    }
    // the box follows the LIVE points: it shrinks when Delete_Point_Boxes drops the part of the map the sensor left
    int box[6];
    FLB_CUDA(h, cudaMemcpyAsync(box, h->bbox_dev.p, sizeof(box), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    for (int k = 0; k < 6; ++k) {
        const int b = box[k] >= 0 ? box[k] : (box[k] ^ 0x7fffffff);
        float f;
        std::memcpy(&f, &b, sizeof(f));
        (k < 3 ? h->map_lo[k] : h->map_hi[k - 3]) = f;
    }
    return rebuild_grid(h, count);
}

// Full path of Add_Points: (existing + new) points sorted by downsample voxel, one thread per voxel, compaction, grid
// rebuilt from scratch.  Taken when a new point lies outside the box the kNN grid covers (the grid has to grow).
static int map_add_points_full(flb_handle* h, const float* st, int n, float downsample_size) {
    const int M = h->M, total = M + n;
    FLB_CUDA(h, h->map_comb.reserve((size_t)total * 3));
    FLB_CUDA(h, h->vkeys.reserve(total));
    FLB_CUDA(h, h->vkeys_sorted.reserve(total));
    FLB_CUDA(h, h->vals.reserve(total));
    FLB_CUDA(h, h->vals_sorted.reserve(total));
    FLB_CUDA(h, h->keep.reserve(total));
    FLB_CUDA(h, h->vox_unclean.reserve(total));
    FLB_CUDA(h, h->vox_rep.reserve(total));
    FLB_CUDA(h, h->vox_counts.reserve(2));
    FLB_CUDA(h, cudaMemsetAsync(h->vox_counts.p, 0, 2 * sizeof(int), h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(h->map_comb.p, h->map_raw.p, (size_t)M * 3 * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(h->map_comb.p + (size_t)M * 3, st, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, h->st_map.mark(h->stream));
    const int nb = (total + 255) / 256;
    {
        LaunchScope ls(h, FAM_OTHER);
        k_vox_keys<<<nb, 256, 0, h->stream>>>(h->map_comb.p, total, downsample_size, h->vkeys.p, h->vals.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    size_t tmp_bytes = 0;
    FLB_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, h->vkeys.p, h->vkeys_sorted.p, h->vals.p, h->vals_sorted.p, total,
                                                0, 63, h->stream));
    FLB_CUDA(h, h->cub_tmp.reserve(tmp_bytes));
    FLB_CUDA(h, cub::DeviceRadixSort::SortPairs(h->cub_tmp.p, tmp_bytes, h->vkeys.p, h->vkeys_sorted.p, h->vals.p, h->vals_sorted.p,
                                                total, 0, 63, h->stream));
    h->launches += 4;
    {
        LaunchScope ls(h, FAM_OTHER);
        k_vox_unclean<<<nb, 256, 0, h->stream>>>(h->vals_sorted.p, h->map_comb.p, total, downsample_size, h->vox_unclean.p,
                                                  h->vox_counts.p);
        k_vox_resolve<<<nb, 256, 0, h->stream>>>(h->vkeys_sorted.p, h->vals_sorted.p, h->map_comb.p, total, M, downsample_size,
                                                  h->vox_unclean.p, h->vox_counts.p, h->vox_rep.p, h->keep.p);
        k_vox_replay<<<1, 1, 0, h->stream>>>(h->vkeys_sorted.p, h->vals_sorted.p, h->map_comb.p, total, downsample_size, h->vox_unclean.p,
                                             h->vox_counts.p, h->vox_rep.p, h->keep.p);
        FLB_CUDA(h, cudaGetLastError());
        h->launches += 2;
    }
    return compact_and_rebuild(h, h->vals_sorted.p, total);
}

static int bits_for(long long span) {
    int b = 1;
    while ((1ll << b) <= span) ++b;
    return b;
}

int flb_map_add_points(flb_handle* h, const float* world_xyz, int n, int stride, float downsample_size) {
    FLB_CHECK_H(h);
    if (h->M <= 0) return fail(h, FLB_ERR_STATE, "flb_map_add_points: no map uploaded");
    if (!world_xyz || n < 0 || stride < 3 || !(downsample_size > 0)) return fail(h, FLB_ERR_INVALID, "flb_map_add_points: bad arguments");
    if (n == 0) return FLB_OK;
    const int M = h->M;
    void* stv = nullptr;
    FLB_CUDA(h, h->st_map.acquire((size_t)n * 3 * sizeof(float), &stv));
    float* st = static_cast<float*>(stv);
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    if (stride == 3) std::memcpy(st, world_xyz, (size_t)n * 3 * sizeof(float));
    else
        for (int i = 0; i < n; ++i) {
            st[3 * (size_t)i] = world_xyz[(size_t)i * stride];
            st[3 * (size_t)i + 1] = world_xyz[(size_t)i * stride + 1];
            st[3 * (size_t)i + 2] = world_xyz[(size_t)i * stride + 2];
        }
    {
        // bounds + finiteness over the packed floats, 24 (= 8 points) at a time into independent accumulators (vectorises)
        float mn[24], mx[24];
        for (int j = 0; j < 24; ++j) { mn[j] = INFINITY; mx[j] = -INFINITY; }
        unsigned bad = 0;
        const size_t n3 = (size_t)n * 3;
        size_t i = 0;
        for (; i + 24 <= n3; i += 24)
            for (int j = 0; j < 24; ++j) {
                const float v = st[i + j];
                unsigned bits;
                std::memcpy(&bits, &v, sizeof(bits));
                bad |= ((bits & 0x7F800000u) == 0x7F800000u) ? 1u : 0u;
                mn[j] = v < mn[j] ? v : mn[j];
                mx[j] = v > mx[j] ? v : mx[j];
            }
        for (; i < n3; ++i) {
            const float v = st[i];
            const int j = (int)(i % 24);
            bad |= std::isfinite(v) ? 0u : 1u;
            mn[j] = v < mn[j] ? v : mn[j];
            mx[j] = v > mx[j] ? v : mx[j];
        }
        if (bad) return fail(h, FLB_ERR_INVALID, "flb_map_add_points: non-finite coordinate");
        for (int j = 0; j < 24; ++j) { lo[j % 3] = std::min(lo[j % 3], mn[j]); hi[j % 3] = std::max(hi[j % 3], mx[j]); }
        const float lim = 1.0e6f * downsample_size;
        for (int k = 0; k < 3; ++k)
            if (lo[k] < -lim || hi[k] > lim) return fail(h, FLB_ERR_INVALID, "flb_map_add_points: coordinate / downsample_size exceeds 2^20 voxels");
    }
    // the input is valid from here on: only now does the map box take it in
    bool inside = true;
    for (int k = 0; k < 3; ++k) inside = inside && lo[k] >= h->grid_lo[k] && hi[k] <= h->grid_hi[k];
    for (int k = 0; k < 3; ++k) { h->map_lo[k] = std::min(h->map_lo[k], lo[k]); h->map_hi[k] = std::max(h->map_hi[k], hi[k]); }
    if (!inside) return map_add_points_full(h, st, n, downsample_size);

    // ---- incremental path: every new point lies inside the box the grid covers
    const GridDesc g = h->grid;
    const int ncell = h->ncell;
    const float ds = downsample_size;
    // voxel keys relative to the grid box, packed into as few bits as the box needs (fewer radix passes)
    const int bx = (int)std::floor(h->grid_lo[0] / ds) - 1, by = (int)std::floor(h->grid_lo[1] / ds) - 1, bz = (int)std::floor(h->grid_lo[2] / ds) - 1;
    const int wx = bits_for((long long)std::floor(h->grid_hi[0] / ds) + 2 - bx), wy = bits_for((long long)std::floor(h->grid_hi[1] / ds) + 2 - by),
              wz = bits_for((long long)std::floor(h->grid_hi[2] / ds) + 2 - bz);
    if (wx + wy + wz > 62) return map_add_points_full(h, st, n, downsample_size);
    FLB_CUDA(h, h->map_comb.reserve((size_t)n * 3));
    FLB_CUDA(h, h->vkeys.reserve(n));
    FLB_CUDA(h, h->vkeys_sorted.reserve(n));
    FLB_CUDA(h, h->vals.reserve(std::max(n, M)));
    FLB_CUDA(h, h->vals_sorted.reserve(std::max(n, M)));
    FLB_CUDA(h, h->keys.reserve(std::max(n, M)));
    FLB_CUDA(h, h->keys_sorted.reserve(std::max(n, M)));
    FLB_CUDA(h, h->dead.reserve(M));
    FLB_CUDA(h, h->ins.reserve(n));
    FLB_CUDA(h, h->dead_before.reserve((size_t)M + 1));
    FLB_CUDA(h, h->merge_counts.reserve(2));
    FLB_CUDA(h, h->map_pts_alt.reserve((size_t)M + n));
    FLB_CUDA(h, h->map_raw_alt.reserve(((size_t)M + n) * 3));
    FLB_CUDA(h, h->cell_start_alt.reserve((size_t)ncell + 1));
    FLB_CUDA(h, h->vox_unclean.reserve(n));
    FLB_CUDA(h, h->vox_rep.reserve(n));
    FLB_CUDA(h, h->vox_counts.reserve(2));
    float* nxyz = h->map_comb.p;
    FLB_CUDA(h, cudaMemcpyAsync(nxyz, st, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, h->st_map.mark(h->stream));
    FLB_CUDA(h, cudaMemsetAsync(h->dead.p, 0, M, h->stream));
    FLB_CUDA(h, cudaMemsetAsync(h->ins.p, 0, n, h->stream));
    FLB_CUDA(h, cudaMemsetAsync(h->vox_counts.p, 0, 2 * sizeof(int), h->stream));
    const int gn = (n + 255) / 256, gm = (M + 255) / 256;
    {
        LaunchScope ls(h, FAM_OTHER);
        k_vox_keys_rel<<<gn, 256, 0, h->stream>>>(nxyz, n, ds, bx, by, bz, wx, wx + wy, h->vkeys.p, h->vals.p, h->vox_unclean.p,
                                                   h->vox_counts.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    size_t tmp_bytes = 0, t2 = 0, t3 = 0;
    int cell_bits = bits_for((long long)ncell);
    FLB_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, h->vkeys.p, h->vkeys_sorted.p, h->vals.p, h->vals_sorted.p, n, 0,
                                                wx + wy + wz, h->stream));
    FLB_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, t2, h->keys.p, h->keys_sorted.p, h->vals.p, h->vals_sorted.p, n, 0, cell_bits, h->stream));
    FLB_CUDA(h, cub::DeviceScan::ExclusiveSum(nullptr, t3, h->dead_before.p, h->dead_before.p, M, h->stream));
    FLB_CUDA(h, h->cub_tmp.reserve(std::max(tmp_bytes, std::max(t2, t3))));
    FLB_CUDA(h, cub::DeviceRadixSort::SortPairs(h->cub_tmp.p, tmp_bytes, h->vkeys.p, h->vkeys_sorted.p, h->vals.p, h->vals_sorted.p, n, 0,
                                                wx + wy + wz, h->stream));
    {
        LaunchScope ls(h, FAM_OTHER);
        k_vox_resolve_incremental<<<gn, 256, 0, h->stream>>>(h->vkeys_sorted.p, h->vals_sorted.p, nxyz, n, ds, g, h->cell_start.p, h->map_pts.p,
                                                              h->vox_unclean.p, h->vox_counts.p, h->vox_rep.p, h->dead.p, h->ins.p);
        k_vox_replay_incremental<<<1, 1, 0, h->stream>>>(nxyz, ds, g, h->cell_start.p, h->map_pts.p, h->vox_counts.p, h->vox_rep.p, h->dead.p,
                                                         h->ins.p);
        h->launches++;
        // inserted points sorted by grid cell (not-inserted ones sort behind every cell)
        k_insert_cells<<<gn, 256, 0, h->stream>>>(nxyz, n, h->ins.p, g, ncell, h->keys.p, h->vals.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    FLB_CUDA(h, cub::DeviceRadixSort::SortPairs(h->cub_tmp.p, t2, h->keys.p, h->keys_sorted.p, h->vals.p, h->vals_sorted.p, n, 0, cell_bits, h->stream));
    {
        LaunchScope ls(h, FAM_OTHER);
        k_dead_to_int<<<gm, 256, 0, h->stream>>>(h->dead.p, M, h->dead_before.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    FLB_CUDA(h, cub::DeviceScan::ExclusiveSum(h->cub_tmp.p, t3, h->dead_before.p, h->dead_before.p, M, h->stream));
    {
        LaunchScope ls(h, FAM_OTHER);
        k_merge_counts<<<1, 32, 0, h->stream>>>(h->dead_before.p, h->dead.p, M, h->keys_sorted.p, n, ncell, h->merge_counts.p);
        k_merge_cell_starts<<<(ncell + 256) / 256, 256, 0, h->stream>>>(h->cell_start.p, h->dead_before.p, h->merge_counts.p, M, h->keys_sorted.p, n,
                                                                         ncell, h->cell_start_alt.p);
        k_merge_existing<<<gm, 256, 0, h->stream>>>(h->map_pts.p, h->dead.p, h->dead_before.p, M, g, h->keys_sorted.p, n, h->map_pts_alt.p,
                                                     h->map_raw_alt.p);
        k_merge_inserts<<<gn, 256, 0, h->stream>>>(nxyz, h->keys_sorted.p, h->vals_sorted.p, n, h->merge_counts.p, h->cell_start_alt.p,
                                                    h->map_pts_alt.p, h->map_raw_alt.p);
        FLB_CUDA(h, cudaGetLastError());
        h->launches += 10;
    }
    int counts[2] = {0, 0};
    FLB_CUDA(h, cudaMemcpyAsync(counts, h->merge_counts.p, sizeof(counts), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    std::swap(h->map_pts, h->map_pts_alt);
    std::swap(h->cell_start, h->cell_start_alt);
    std::swap(h->map_raw, h->map_raw_alt);
    h->M = M - counts[0] + counts[1];
    h->last_pass_valid = false;
    return FLB_OK;
}

int flb_map_delete_boxes(flb_handle* h, const float* boxes, int nb) {
    FLB_CHECK_H(h);
    if (h->M <= 0) return fail(h, FLB_ERR_STATE, "flb_map_delete_boxes: no map uploaded");
    if (nb < 0 || (nb > 0 && !boxes)) return fail(h, FLB_ERR_INVALID, "flb_map_delete_boxes: bad arguments");
    if (nb == 0) return FLB_OK;
    const int M = h->M;
    void* stv = nullptr;
    FLB_CUDA(h, h->st_misc.acquire((size_t)nb * 6 * sizeof(float), &stv));
    std::memcpy(stv, boxes, (size_t)nb * 6 * sizeof(float));
    FLB_CUDA(h, h->boxes.reserve((size_t)nb * 6));
    FLB_CUDA(h, cudaMemcpyAsync(h->boxes.p, stv, (size_t)nb * 6 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, h->st_misc.mark(h->stream));
    FLB_CUDA(h, h->map_comb.reserve((size_t)M * 3));
    FLB_CUDA(h, h->vals.reserve(M));
    FLB_CUDA(h, h->keep.reserve(M));
    FLB_CUDA(h, cudaMemcpyAsync(h->map_comb.p, h->map_raw.p, (size_t)M * 3 * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
    {
        LaunchScope ls(h, FAM_OTHER);
        k_box_flags<<<(M + 255) / 256, 256, 0, h->stream>>>(h->map_comb.p, M, h->boxes.p, nb, h->keep.p, h->vals.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    return compact_and_rebuild(h, h->vals.p, M);
}

int flb_map_size(const flb_handle* h) { return h ? h->M : 0; }

int flb_map_download(flb_handle* h, float* xyz, int capacity, int* M_out) {
    FLB_CHECK_H(h);
    if (M_out) *M_out = h->M;
    if (!xyz || capacity <= 0) return FLB_OK;
    const int n = std::min(capacity, h->M);
    FLB_CUDA(h, cudaMemcpyAsync(xyz, h->map_raw.p, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    return FLB_OK;
}

int flb_imu_undistort(flb_handle* h, const flb_imu_params* prm, flb_imu_carry* carry, const flb_imu_sample* v_imu, int n_imu,
                      double pcl_beg_time, double pcl_end_time, const float* pts, int stride, int offset_index, int n_points,
                      float* out_xyz, double* poses_out, int* n_poses_out) {
    FLB_CHECK_H(h);
    if (!prm || !carry || !v_imu || n_imu < 1 || n_points < 0 || (n_points > 0 && (!pts || !out_xyz)) || stride < 4 ||
        offset_index < 3 || offset_index >= stride)
        return fail(h, FLB_ERR_INVALID, "flb_imu_undistort: bad arguments");
    if (!h->state_valid) return fail(h, FLB_ERR_STATE, "flb_imu_undistort: no device state (flb_state_upload)");
    { int rcf = flush_state_ops(h); if (rcf) return rcf; }
    for (int i = 0; i + 1 < n_imu; ++i)
        if (!(v_imu[i + 1].t >= v_imu[i].t)) return fail(h, FLB_ERR_INVALID, "flb_imu_undistort: IMU times must be non-decreasing");
    static_assert(sizeof(ImuSampleDev) == sizeof(flb_imu_sample) && sizeof(ImuCarryDev) == sizeof(flb_imu_carry), "ABI layout");
    static_assert(sizeof(ImuPose) == 22 * sizeof(double), "IMUpose layout");
    ImuParamsDev d;
    std::memcpy(d.cov_gyr, prm->cov_gyr, sizeof(d.cov_gyr));
    std::memcpy(d.cov_acc, prm->cov_acc, sizeof(d.cov_acc));
    std::memcpy(d.cov_bias_gyr, prm->cov_bias_gyr, sizeof(d.cov_bias_gyr));
    std::memcpy(d.cov_bias_acc, prm->cov_bias_acc, sizeof(d.cov_bias_acc));
    d.G_m_s2 = prm->G_m_s2;
    d.mean_acc_norm = prm->mean_acc_norm;
    std::memcpy(d.R_LI, prm->R_LI, sizeof(d.R_LI));
    std::memcpy(d.t_LI, prm->t_LI, sizeof(d.t_LI));
    const size_t n1 = (size_t)std::max(n_points, 1);
    // device buffers: samples + carry + aux + poses packed in one double array, points as float4 in/out
    const size_t off_carry = (size_t)n_imu * 7, off_aux = off_carry + 7, off_poses = off_aux + 16, total = off_poses + (size_t)n_imu * 22;
    FLB_CUDA(h, h->imu_buf.reserve(total));
    FLB_CUDA(h, h->imu_pts.reserve(n1 * 2));
    FLB_CUDA(h, h->imu_heads.reserve(n1));
    void* stv = nullptr;
    FLB_CUDA(h, h->st_scan.acquire(n1 * 4 * sizeof(float) + (off_aux) * sizeof(double), &stv));
    double* st_d = static_cast<double*>(stv);
    std::memcpy(st_d, v_imu, (size_t)n_imu * sizeof(flb_imu_sample));
    std::memcpy(st_d + off_carry, carry, sizeof(flb_imu_carry));
    float* st_p = reinterpret_cast<float*>(st_d + off_aux);
    for (int i = 0; i < n_points; ++i) {
        st_p[4 * (size_t)i] = pts[(size_t)i * stride];
        st_p[4 * (size_t)i + 1] = pts[(size_t)i * stride + 1];
        st_p[4 * (size_t)i + 2] = pts[(size_t)i * stride + 2];
        st_p[4 * (size_t)i + 3] = pts[(size_t)i * stride + offset_index];
    }
    FLB_CUDA(h, cudaMemcpyAsync(h->imu_buf.p, st_d, off_aux * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    float4* d_in = h->imu_pts.p;
    float4* d_out = h->imu_pts.p + n1;
    if (n_points > 0)
        FLB_CUDA(h, cudaMemcpyAsync(d_in, st_p, (size_t)n_points * 4 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, h->st_scan.mark(h->stream));
    const ImuSampleDev* d_imu = reinterpret_cast<const ImuSampleDev*>(h->imu_buf.p);
    ImuCarryDev* d_carry = reinterpret_cast<ImuCarryDev*>(h->imu_buf.p + off_carry);
    ImuAux* d_aux = reinterpret_cast<ImuAux*>(h->imu_buf.p + off_aux);
    ImuPose* d_poses = reinterpret_cast<ImuPose*>(h->imu_buf.p + off_poses);
    {
        LaunchScope ls(h, FAM_OTHER);
        k_imu_propagate<<<1, 352, 0, h->stream>>>(&h->states.p[0], d_imu, n_imu, d, pcl_beg_time, pcl_end_time, d_carry, d_poses, d_aux);
        FLB_CUDA(h, cudaGetLastError());
    }
    if (n_points > 0) {                                                           // :776
        const int g = (n_points + 255) / 256;
        const float* in_f = reinterpret_cast<const float*>(d_in);
        LaunchScope ls(h, FAM_OTHER);
        k_imu_heads<<<g, 256, 0, h->stream>>>(in_f + 3, 4, n_points, d_poses, d_aux, h->imu_heads.p);
        k_suffix_min<<<1, 1024, 0, h->stream>>>(h->imu_heads.p, n_points);
        k_imu_undistort<<<g, 256, 0, h->stream>>>(in_f, 4, in_f + 3, 4, n_points, d_poses, d_aux, h->imu_heads.p, d, d_out);
        FLB_CUDA(h, cudaGetLastError());
        h->launches += 2;
    }
    // results: carry, aux (n_poses), poses, points
    const size_t out_bytes = (7 + 16 + (size_t)n_imu * 22) * sizeof(double) + n1 * 4 * sizeof(float);
    FLB_CUDA(h, h->pin_out.reserve(out_bytes));
    char* po = static_cast<char*>(h->pin_out.p);
    FLB_CUDA(h, cudaMemcpyAsync(po, h->imu_buf.p + off_carry, (7 + 16 + (size_t)n_imu * 22) * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    float* po_pts = reinterpret_cast<float*>(po + (7 + 16 + (size_t)n_imu * 22) * sizeof(double));
    if (n_points > 0)
        FLB_CUDA(h, cudaMemcpyAsync(po_pts, d_out, (size_t)n_points * 4 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    std::memcpy(carry, po, sizeof(flb_imu_carry));
    ImuAux aux;
    std::memcpy(&aux, po + 7 * sizeof(double), sizeof(aux));
    if (n_poses_out) *n_poses_out = aux.n_poses;
    if (poses_out) std::memcpy(poses_out, po + (7 + 16) * sizeof(double), (size_t)aux.n_poses * 22 * sizeof(double));
    for (int i = 0; i < n_points; ++i) {
        out_xyz[3 * (size_t)i] = po_pts[4 * (size_t)i];
        out_xyz[3 * (size_t)i + 1] = po_pts[4 * (size_t)i + 1];
        out_xyz[3 * (size_t)i + 2] = po_pts[4 * (size_t)i + 2];
    }
    h->last_pass_valid = false;
    h->last_vio_valid = false;
    return FLB_OK;
}

int flb_visual_candidates(flb_handle* h, const double Rcw[9], const double Pcw[3], const float* world_xyz, int n, int stride,
                          int grid_size, int border, float* map_value, int* winner) {
    FLB_CHECK_H(h);
    if (!Rcw || !Pcw || n < 0 || (n > 0 && !world_xyz) || stride < 3 || grid_size < 1 || border < 0 || !map_value || !winner)
        return fail(h, FLB_ERR_INVALID, "flb_visual_candidates: bad arguments");
    if (!h->cam_set || h->img_w <= 0) return fail(h, FLB_ERR_STATE, "flb_visual_candidates: camera and image must be set first");
    const int gw = h->img_w / grid_size, gh = h->img_h / grid_size, ncell = gw * gh;      // :55-57
    if (ncell < 1) return fail(h, FLB_ERR_INVALID, "flb_visual_candidates: grid_size larger than the image");
    { int rcq = vio_inputs_acquire(h); if (rcq) return rcq; }                           // the image upload has landed
    const size_t n1 = (size_t)std::max(n, 1);
    FLB_CUDA(h, h->vm_key.reserve((size_t)ncell));
    FLB_CUDA(h, h->vm_val.reserve((size_t)ncell));
    FLB_CUDA(h, h->vm_win.reserve((size_t)ncell));
    FLB_CUDA(h, h->vm_pts.reserve(n1 * 3));
    FLB_CUDA(h, h->vm_pose.reserve(12));
    void* stv = nullptr;
    const size_t st_bytes = n1 * 3 * sizeof(float) + (size_t)ncell * sizeof(float) + 12 * sizeof(double);
    FLB_CUDA(h, h->st_scan.acquire(st_bytes, &stv));
    double* st_pose = static_cast<double*>(stv);
    std::memcpy(st_pose, Rcw, 9 * sizeof(double));
    std::memcpy(st_pose + 9, Pcw, 3 * sizeof(double));
    float* st_val = reinterpret_cast<float*>(st_pose + 12);
    std::memcpy(st_val, map_value, (size_t)ncell * sizeof(float));
    float* st_pts = st_val + ncell;
    for (int i = 0; i < n; ++i) {
        st_pts[3 * (size_t)i] = world_xyz[(size_t)i * stride];
        st_pts[3 * (size_t)i + 1] = world_xyz[(size_t)i * stride + 1];
        st_pts[3 * (size_t)i + 2] = world_xyz[(size_t)i * stride + 2];
    }
    FLB_CUDA(h, cudaMemcpyAsync(h->vm_pose.p, st_pose, 12 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(h->vm_val.p, st_val, (size_t)ncell * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    if (n > 0) FLB_CUDA(h, cudaMemcpyAsync(h->vm_pts.p, st_pts, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, h->st_scan.mark(h->stream));
    {
        LaunchScope ls(h, FAM_OTHER);
        k_vmap_seed<<<(ncell + 255) / 256, 256, 0, h->stream>>>(h->vm_val.p, ncell, h->vm_key.p);
        if (n > 0)
            k_vmap_candidates<<<(n + 127) / 128, 128, 0, h->stream>>>(h->cam, h->vm_pose.p, h->img.p, h->vm_pts.p, n, grid_size, gh, border,
                                                                      h->vm_key.p);
        k_vmap_resolve<<<(ncell + 255) / 256, 256, 0, h->stream>>>(h->vm_key.p, ncell, h->vm_val.p, h->vm_win.p);
        FLB_CUDA(h, cudaGetLastError());
        h->launches += 2;
    }
    FLB_CUDA(h, h->pin_out.reserve((size_t)ncell * (sizeof(float) + sizeof(int))));
    char* po = static_cast<char*>(h->pin_out.p);
    FLB_CUDA(h, cudaMemcpyAsync(po, h->vm_val.p, (size_t)ncell * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(po + (size_t)ncell * sizeof(float), h->vm_win.p, (size_t)ncell * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    std::memcpy(map_value, po, (size_t)ncell * sizeof(float));
    std::memcpy(winner, po + (size_t)ncell * sizeof(float), (size_t)ncell * sizeof(int));
    return vio_inputs_release(h);
}

int flb_voxel_grid(flb_handle* h, const float* xyz, int n, int stride, float leaf, float* out_xyz, int capacity, int* n_out) {
    FLB_CHECK_H(h);
    if (n < 0 || (n > 0 && !xyz) || stride < 3 || !(leaf > 0) || !n_out || capacity < 0 || (capacity > 0 && !out_xyz))
        return fail(h, FLB_ERR_INVALID, "flb_voxel_grid: bad arguments");
    *n_out = 0;
    if (n == 0) return FLB_OK;
    void* stv = nullptr;
    FLB_CUDA(h, h->st_scan.acquire((size_t)n * 3 * sizeof(float), &stv));
    float* st = static_cast<float*>(stv);
    for (int i = 0; i < n; ++i)
        for (int k = 0; k < 3; ++k) {
            const float v = xyz[(size_t)i * stride + k];
            if (!std::isfinite(v)) return fail(h, FLB_ERR_INVALID, "flb_voxel_grid: non-finite coordinate at point %d", i);
            st[3 * (size_t)i + k] = v;
        }
    FLB_CUDA(h, h->scan_raw.reserve((size_t)n * 3));
    FLB_CUDA(h, h->skeys.reserve(n));
    FLB_CUDA(h, h->skeys_sorted.reserve(n));
    FLB_CUDA(h, h->svals.reserve(n));
    FLB_CUDA(h, h->svals_sorted.reserve(n));
    FLB_CUDA(h, h->dead_before.reserve((size_t)2 * n + 2));      // head flags | ranks
    FLB_CUDA(h, h->map_comb.reserve((size_t)n * 3));             // centroids
    FLB_CUDA(h, h->bbox_dev.reserve(8));
    int* head = h->dead_before.p;
    int* rank = h->dead_before.p + n;
    const int init[8] = {0x7fffffff, 0x7fffffff, 0x7fffffff, (int)0x80000000, (int)0x80000000, (int)0x80000000, 0, 0};
    FLB_CUDA(h, cudaMemcpyAsync(h->bbox_dev.p, init, sizeof(init), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(h->scan_raw.p, st, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, h->st_scan.mark(h->stream));
    const float inv_leaf = 1.0f / leaf;                              // inverse_leaf_size_ = Array4f::Ones() / leaf_size_
    const int g = (n + 255) / 256;
    {
        LaunchScope ls(h, FAM_OTHER);
        k_bbox<<<std::min(g, 4 * std::max(h->num_sms, 1)), 256, 0, h->stream>>>(h->scan_raw.p, n, h->bbox_dev.p);
        k_vg_keys<<<g, 256, 0, h->stream>>>(h->scan_raw.p, n, h->bbox_dev.p, inv_leaf, h->skeys.p, h->svals.p, h->bbox_dev.p + 6);
        FLB_CUDA(h, cudaGetLastError());
    }
    size_t t1 = 0, t2 = 0;
    FLB_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, t1, h->skeys.p, h->skeys_sorted.p, h->svals.p, h->svals_sorted.p, n, 0, 31, h->stream));
    FLB_CUDA(h, cub::DeviceScan::ExclusiveSum(nullptr, t2, head, rank, n, h->stream));
    FLB_CUDA(h, h->cub_tmp.reserve(std::max(t1, t2)));
    FLB_CUDA(h, cub::DeviceRadixSort::SortPairs(h->cub_tmp.p, t1, h->skeys.p, h->skeys_sorted.p, h->svals.p, h->svals_sorted.p, n, 0, 31, h->stream));
    {
        LaunchScope ls(h, FAM_OTHER);
        k_vg_heads<<<g, 256, 0, h->stream>>>(h->skeys_sorted.p, n, head);
        FLB_CUDA(h, cudaGetLastError());
    }
    FLB_CUDA(h, cub::DeviceScan::ExclusiveSum(h->cub_tmp.p, t2, head, rank, n, h->stream));
    {
        LaunchScope ls(h, FAM_OTHER);
        k_vg_centroids<<<g, 256, 0, h->stream>>>(h->scan_raw.p, h->skeys_sorted.p, h->svals_sorted.p, head, rank, n, h->map_comb.p,
                                                  h->bbox_dev.p + 7);
        FLB_CUDA(h, cudaGetLastError());
        h->launches += 8;
    }
    int tail[2] = {0, 0};
    FLB_CUDA(h, cudaMemcpyAsync(tail, h->bbox_dev.p + 6, sizeof(tail), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    if (tail[0]) return fail(h, FLB_ERR_INVALID, "flb_voxel_grid: leaf size too small for the cloud's extent (index overflow, as PCL warns)");
    *n_out = tail[1];
    const int m = std::min(tail[1], capacity);
    if (m > 0) {
        FLB_CUDA(h, cudaMemcpyAsync(out_xyz, h->map_comb.p, (size_t)m * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
        FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    }
    h->N = 0;                                    // the scan slot was used as scratch
    h->last_pass_valid = false;
    return FLB_OK;
}

int flb_scan_upload(flb_handle* h, const float* body_xyz, int N, int stride) {
    FLB_CHECK_H(h);
    if ((!body_xyz && N != 0) || N < 0 || stride < 3) return fail(h, FLB_ERR_INVALID, "flb_scan_upload: bad arguments");
    const size_t n1 = (size_t)std::max(N, 1);
    void* stv = nullptr;
    FLB_CUDA(h, h->st_scan.acquire(n1 * 3 * sizeof(float), &stv));
    float* st = static_cast<float*>(stv);
    float lo[3] = {INFINITY, INFINITY, INFINITY};
    const bool direct = N > 0 && stride == 3 && is_pinned(body_xyz);      // page-locked packed source: no staging copy
    if (direct) st = const_cast<float*>(body_xyz);
    else if (stride == 3) std::memcpy(st, body_xyz, (size_t)N * 3 * sizeof(float));
    else
        for (int i = 0; i < N; ++i) {
            st[3 * (size_t)i] = body_xyz[(size_t)i * stride];
            st[3 * (size_t)i + 1] = body_xyz[(size_t)i * stride + 1];
            st[3 * (size_t)i + 2] = body_xyz[(size_t)i * stride + 2];
        }
    {
        // bounds + finiteness over the packed floats, 24 (= 8 points) at a time into 24 independent accumulators:
        // no cross-iteration dependency, so the host compiler vectorises the inner loop as it stands
        float mn[24];
        for (int j = 0; j < 24; ++j) mn[j] = INFINITY;
        unsigned bad = 0;
        const size_t n3 = (size_t)N * 3;
        size_t i = 0;
        for (; i + 24 <= n3; i += 24)
            for (int j = 0; j < 24; ++j) {
                const float v = st[i + j];
                unsigned bits;
                std::memcpy(&bits, &v, sizeof(bits));
                bad |= ((bits & 0x7F800000u) == 0x7F800000u) ? 1u : 0u;
                mn[j] = v < mn[j] ? v : mn[j];
            }
        for (; i < n3; ++i) {
            const float v = st[i];
            const int j = (int)(i % 24);
            bad |= std::isfinite(v) ? 0u : 1u;
            mn[j] = v < mn[j] ? v : mn[j];
        }
        for (int j = 0; j < 24; ++j) lo[j % 3] = std::min(lo[j % 3], mn[j]);
        if (bad) return fail(h, FLB_ERR_INVALID, "flb_scan_upload: non-finite coordinate");
    }
    // The copy and the ordering run on `scan_stream` into the slot that is NOT being read: updates of the previous frame
    // still queued or running on `stream` keep their scan, and -- because the persistent kernels leave one SM free and
    // the ordering is one block (k_scan_sort_block) -- this frame's upload overlaps them instead of queueing behind them.
    const int cur = h->scan_slot, alt = cur ^ 1;
    cudaStream_t ss = h->scan_stream;
    FLB_CUDA(h, cudaEventRecord(h->ev_scan_free[cur], h->stream));     // all readers of the current slot are enqueued before this
    h->scan_free_valid[cur] = true;
    if (h->scan_free_valid[alt]) FLB_CUDA(h, cudaStreamWaitEvent(ss, h->ev_scan_free[alt], 0));
    // (scan_raw / skeys / svals double as flb_voxel_grid's scratch on `stream`; that call ends with a stream synchronise)
    FLB_CUDA(h, h->scan_raw.reserve(n1 * 3));
    FLB_CUDA(h, h->scan_alt.reserve(n1));
    FLB_CUDA(h, h->sel_alt.reserve(n1));
    FLB_CUDA(h, h->plane_ok_alt.reserve(n1));
    FLB_CUDA(h, h->plane_alt.reserve(n1));
    const size_t nb = (n1 + kLioBlock - 1) / kLioBlock;
    FLB_CUDA(h, h->partials.reserve(std::max<size_t>(nb * lio_packed(12), h->partials.cap)));
    bool flags_done = false;
    if (N > 0) {
        FLB_CUDA(h, cudaMemcpyAsync(h->scan_raw.p, st, (size_t)N * 3 * sizeof(float), cudaMemcpyHostToDevice, ss));
        if (!direct) FLB_CUDA(h, h->st_scan.mark(ss));
        // Morton order in the body frame (cell = twice the map grid's cell): spatially coherent warps at any pose
        const float inv_cell = 0.5f / (float)h->cfg.cell_size;
        // One-block ordering vs keys + device-wide radix sort + gather (identical order).  Measured on an idle GPU
        // (profiles/scan_upload_probe.py, copy included): 8 k points 45 vs 76 us, 16 k 78 vs 82, 24 k 116 vs 89 -- but the
        // one-block kernel runs on the SM the persistent kernels leave free, so when an update is still running on
        // `stream` (a pipelined caller) it costs nothing, while the device-wide kernels would queue behind the update.
        // So: one block up to 16 896 points always, up to 25 600 when `stream` is busy; FLB_BLOCK_SORT=0 / 2 or
        // flb_debug_set_scan_sort force the device-wide / one-block path.
        static const int env_block_sort = [] { const char* e = getenv("FLB_BLOCK_SORT"); return e ? atoi(e) : 1; }();
        const int mode = h->scan_sort_mode ? h->scan_sort_mode : (env_block_sort == 0 ? 2 : (env_block_sort == 2 ? 1 : 0));
        bool use_block = N <= 1024 * 25 && mode != 2;
        if (use_block && mode == 0 && N > 512 * 33) {
            const cudaError_t q = cudaStreamQuery(h->stream);
            (void)cudaGetLastError();
            use_block = (q == cudaErrorNotReady);
        }
        if (use_block) {
            LaunchScope ls(h, FAM_OTHER);
            int rcs = N <= 512 * 17   ? launch_scan_sort_block<512, 17>(h, ss, N, lo, inv_cell)
                      : N <= 512 * 33 ? launch_scan_sort_block<512, 33>(h, ss, N, lo, inv_cell)
                                      : launch_scan_sort_block<1024, 25>(h, ss, N, lo, inv_cell);
            if (rcs) return rcs;
            flags_done = true;
        } else {
            FLB_CUDA(h, h->skeys.reserve(n1));
            FLB_CUDA(h, h->skeys_sorted.reserve(n1));
            FLB_CUDA(h, h->svals.reserve(n1));
            FLB_CUDA(h, h->svals_sorted.reserve(n1));
            const int g = (N + 255) / 256;
            {
                LaunchScope ls(h, FAM_OTHER);
                k_scan_keys<<<g, 256, 0, ss>>>(h->scan_raw.p, N, lo[0], lo[1], lo[2], inv_cell, h->skeys.p, h->svals.p);
                FLB_CUDA(h, cudaGetLastError());
            }
            size_t tmp_bytes = 0;
            FLB_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, h->skeys.p, h->skeys_sorted.p, h->svals.p,
                                                        h->svals_sorted.p, N, 0, 24, ss));
            FLB_CUDA(h, h->scan_cub_tmp.reserve(tmp_bytes));
            FLB_CUDA(h, cub::DeviceRadixSort::SortPairs(h->scan_cub_tmp.p, tmp_bytes, h->skeys.p, h->skeys_sorted.p, h->svals.p,
                                                        h->svals_sorted.p, N, 0, 24, ss));
            h->launches += 3;
            {
                LaunchScope ls(h, FAM_OTHER);
                k_scan_gather<<<g, 256, 0, ss>>>(h->scan_raw.p, N, h->svals_sorted.p, h->scan_alt.p);
                FLB_CUDA(h, cudaGetLastError());
            }
        }
    }
    if (!flags_done) {
        // point_selected_surf.resize(N, true) (src/laserMapping.cpp:1469)
        FLB_CUDA(h, cudaMemsetAsync(h->sel_alt.p, 1, n1, ss));
        FLB_CUDA(h, cudaMemsetAsync(h->plane_ok_alt.p, 0, n1, ss));
    }
    FLB_CUDA(h, cudaEventRecord(h->ev_scan_ready, ss));
    FLB_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_scan_ready, 0));
    std::swap(h->scan, h->scan_alt);
    std::swap(h->sel, h->sel_alt);
    std::swap(h->plane_ok, h->plane_ok_alt);
    std::swap(h->plane, h->plane_alt);
    h->scan_slot = alt;
    h->N = N;     // enqueue-only: everything later on this handle's stream is ordered after the upload
    h->last_pass_valid = false;
    return FLB_OK;
}

int flb_knn(flb_handle* h, const float* q, int nq, int* idx, float* d2) {
    FLB_CHECK_H(h);
    if (h->M <= 0) return fail(h, FLB_ERR_STATE, "flb_knn: no map uploaded");
    if (!q || !idx || !d2 || nq < 0) return fail(h, FLB_ERR_INVALID, "flb_knn: bad arguments");
    if (nq == 0) return FLB_OK;
    DevBuf<float> dq, dd;
    DevBuf<int> di;
    FLB_CUDA(h, dq.reserve((size_t)nq * 3));
    FLB_CUDA(h, dd.reserve((size_t)nq * kMatch));
    FLB_CUDA(h, di.reserve((size_t)nq * kMatch));
    FLB_CUDA(h, cudaMemcpyAsync(dq.p, q, (size_t)nq * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    {
        LaunchScope ls(h, FAM_LIO_KNN);
        k_knn<<<(nq + 127) / 128, 128, 0, h->stream>>>(h->grid, h->cell_start.p, h->map_pts.p, dq.p, nq, di.p, dd.p);
    }
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(idx, di.p, (size_t)nq * kMatch * sizeof(int), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d2, dd.p, (size_t)nq * kMatch * sizeof(float), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    dq.release(); dd.release(); di.release();
    if (e != cudaSuccess) return fail(h, FLB_ERR_CUDA, "flb_knn: %s", cudaGetErrorString(e));
    return FLB_OK;
}

// ---------------------------------------------------------------------------------------
int flb_lio_pass(flb_handle* h, const flb_lio_params* prm, const double R[9], const double p[3], int rematch, int width,
                 flb_normal_eq* out) {
    FLB_CHECK_H(h);
    if (!prm || !R || !p || !out || (width != 6 && width != 12)) return fail(h, FLB_ERR_INVALID, "flb_lio_pass: bad arguments");
    if (h->M <= 0 || h->N <= 0) return fail(h, FLB_ERR_STATE, "flb_lio_pass: map and scan must be uploaded first");
    const int N = h->N;
    FLB_CUDA(h, h->x_world.reserve((size_t)N * 3));
    FLB_CUDA(h, h->x_nn_idx.reserve((size_t)N * kMatch));
    FLB_CUDA(h, h->x_nn_d2.reserve((size_t)N * kMatch));
    FLB_CUDA(h, h->x_pd2.reserve(N));
    FLB_CUDA(h, h->x_pabcd.reserve((size_t)N * 4));
    FLB_CUDA(h, h->x_rowmask.reserve(N));
    FLB_CUDA(h, h->x_rows.reserve((size_t)N * 12));
    FLB_CUDA(h, h->x_meas.reserve(N));
    LioParamsDev d;
    to_dev_params(prm, d);
    void* stv = nullptr;
    FLB_CUDA(h, h->st_misc.acquire(12 * sizeof(double), &stv));
    double* st = static_cast<double*>(stv);
    std::memcpy(st, R, 9 * sizeof(double));
    std::memcpy(st + 9, p, 3 * sizeof(double));
    FLB_CUDA(h, cudaMemcpyAsync(h->pose12.p, st, 12 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, h->st_misc.mark(h->stream));
    LioArgs a = make_lio_args(h, d, true, width);
    a.force_rematch = rematch ? 1 : 0;
    a.pose_override = h->pose12.p;
    int rc = launch_lio_pass(h, a, width, rematch != 0);
    if (rc) return rc;
    const int K = lio_packed(width);
    if (h->comm) {
        rc = allreduce_packed(h, h->partials.p, lio_nblocks(h), K);
        if (rc) return rc;
    } else {
        LaunchScope ls(h, FAM_SOLVE);
        k_reduce_only<<<1, 32, 0, h->stream>>>(h->partials.p, lio_nblocks(h), K, h->packed.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    double* po = static_cast<double*>(h->pin_out.p);
    FLB_CUDA(h, cudaMemcpyAsync(po, h->packed.p, K * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    std::memset(out, 0, sizeof(*out));
    out->width = width;
    int k = 0;
    for (int r = 0; r < width; ++r)
        for (int c = r; c < width; ++c) {
            out->HTH[r * width + c] = po[k];
            out->HTH[c * width + r] = po[k];
            ++k;
        }
    for (int r = 0; r < width; ++r) out->HTh[r] = po[k + r];
    out->n_eff = (int)po[K - 2];
    out->sum_abs_res = po[K - 1];
    h->last_pass_width = width;
    h->last_pass_valid = true;
    return FLB_OK;
}

int flb_lio_export(flb_handle* h, float* world_xyz, int* nn_idx, float* nn_d2, float* pabcd, float* pd2, uint8_t* selected,
                   double* rows, double* meas, int* sel_idx, int* n_rows) {
    FLB_CHECK_H(h);
    if (!h->last_pass_valid) return fail(h, FLB_ERR_STATE, "flb_lio_export: no flb_lio_pass to export");
    const int N = h->N, W = h->last_pass_width;
    cudaStream_t s = h->stream;
    if (world_xyz) FLB_CUDA(h, cudaMemcpyAsync(world_xyz, h->x_world.p, (size_t)N * 3 * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (nn_idx) FLB_CUDA(h, cudaMemcpyAsync(nn_idx, h->x_nn_idx.p, (size_t)N * kMatch * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (nn_d2) FLB_CUDA(h, cudaMemcpyAsync(nn_d2, h->x_nn_d2.p, (size_t)N * kMatch * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (pabcd) FLB_CUDA(h, cudaMemcpyAsync(pabcd, h->x_pabcd.p, (size_t)N * 4 * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (pd2) FLB_CUDA(h, cudaMemcpyAsync(pd2, h->x_pd2.p, (size_t)N * sizeof(float), cudaMemcpyDeviceToHost, s));
    std::vector<unsigned char> mask(N);
    FLB_CUDA(h, cudaMemcpyAsync(mask.data(), h->x_rowmask.p, N, cudaMemcpyDeviceToHost, s));
    std::vector<double> hrows, hmeas;
    if (rows || meas) {
        hrows.resize((size_t)N * W);
        hmeas.resize(N);
        FLB_CUDA(h, cudaMemcpyAsync(hrows.data(), h->x_rows.p, (size_t)N * W * sizeof(double), cudaMemcpyDeviceToHost, s));
        FLB_CUDA(h, cudaMemcpyAsync(hmeas.data(), h->x_meas.p, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    FLB_CUDA(h, cudaStreamSynchronize(s));
    // order-preserving compaction == laserCloudOri / corr_normvect (src/laserMapping.cpp:1588-1600)
    int n = 0;
    for (int i = 0; i < N; ++i) {
        if (selected) selected[i] = mask[i];
        if (!mask[i]) continue;
        if (rows) std::memcpy(rows + (size_t)n * W, hrows.data() + (size_t)i * W, W * sizeof(double));
        if (meas) meas[n] = hmeas[i];
        if (sel_idx) sel_idx[n] = i;
        ++n;
    }
    if (n_rows) *n_rows = n;
    return FLB_OK;
}

int flb_state_upload(flb_handle* h, const flb_state18* x, const flb_state18* x_prop) {
    FLB_CHECK_H(h);
    if (!x || !x_prop) return fail(h, FLB_ERR_INVALID, "flb_state_upload: null state");
    void* stv = nullptr;
    FLB_CUDA(h, h->st_state.acquire(2 * sizeof(State18), &stv));
    State18* st = static_cast<State18*>(stv);
    std::memcpy(&st[0], x, sizeof(State18));
    std::memcpy(&st[1], x_prop, sizeof(State18));
    {
        void* dsrc = nullptr;
        FLB_CUDA(h, cudaHostGetDevicePointer(&dsrc, st, 0));
        LaunchScope ls(h, FAM_OTHER);
        k_state_install<<<1, 256, 0, h->stream>>>(static_cast<const double*>(dsrc), h->states.p);   // [0..1] and the saved pair [3..4]
        FLB_CUDA(h, cudaGetLastError());
    }
    FLB_CUDA(h, h->st_state.mark(h->stream));
    h->state_valid = true;
    h->reset_pending = h->prior_pending = false;     // both superseded by the upload
    return FLB_OK;
}

int flb_state_reset_enqueue(flb_handle* h) {
    FLB_CHECK_H(h);
    if (!h->state_valid) return fail(h, FLB_ERR_STATE, "flb_state_reset_enqueue: no state uploaded");
    h->prior_pending = false;            // overwritten by the reset
    h->reset_pending = true;             // performed by the next LIO kernel (or flushed as a copy by any other consumer)
    return FLB_OK;
}

int flb_state_set_prior_enqueue(flb_handle* h) {
    FLB_CHECK_H(h);
    if (!h->state_valid) return fail(h, FLB_ERR_STATE, "flb_state_set_prior_enqueue: no state uploaded");
    { int rcf = flush_state_ops(h); if (rcf) return rcf; }      // an earlier pending reset / prior comes first
    h->prior_pending = true;             // performed by the next VIO kernel (or flushed as a copy by any other consumer)
    return FLB_OK;
}

int flb_state_download(flb_handle* h, flb_state18* x, flb_lio_report* lio, flb_vio_report* vio) {
    FLB_CHECK_H(h);
    if (!h->state_valid) return fail(h, FLB_ERR_STATE, "flb_state_download: no state uploaded");
    { int rcf = flush_state_ops(h); if (rcf) return rcf; }
    char* po = static_cast<char*>(h->pin_out.p);
    FLB_CUDA(h, cudaMemcpyAsync(po, &h->states.p[0], sizeof(State18), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(po + sizeof(State18), h->lio_ctrl.p, sizeof(LioCtrl), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(po + sizeof(State18) + sizeof(LioCtrl), h->vio_ctrl.p, sizeof(VioCtrl), cudaMemcpyDeviceToHost,
                                h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(po + sizeof(State18) + sizeof(LioCtrl) + sizeof(VioCtrl), h->barrier.p, sizeof(GridBarrier),
                                cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    {
        GridBarrier b;
        std::memcpy(&b, po + sizeof(State18) + sizeof(LioCtrl) + sizeof(VioCtrl), sizeof(b));
        if (b.timeout) {
            cudaMemset(h->barrier.p, 0, sizeof(GridBarrier));
            return fail(h, FLB_ERR_TIMEOUT, "device-side grid barrier watchdog tripped");
        }
    }
    if (x) std::memcpy(x, po, sizeof(State18));
    if (lio) {
        LioCtrl c;
        std::memcpy(&c, po + sizeof(State18), sizeof(c));
        fill_lio_report(c, lio);
    }
    if (vio) {
        VioCtrl c;
        std::memcpy(&c, po + sizeof(State18) + sizeof(LioCtrl), sizeof(c));
        fill_vio_report(c, vio);
    }
    return FLB_OK;
}

// Pipelined result read-back: enqueue the copy of (state, reports) of everything enqueued so far into result slot
// `slot`, return at once; flb_state_download_wait blocks on that slot only, so frame k's result can be collected while
// frame k+1 is already uploading / running.
int flb_state_download_enqueue(flb_handle* h, int slot) {
    FLB_CHECK_H(h);
    if (slot < 0 || slot > 1) return fail(h, FLB_ERR_INVALID, "flb_state_download_enqueue: slot must be 0 or 1");
    if (!h->state_valid) return fail(h, FLB_ERR_STATE, "flb_state_download_enqueue: no state uploaded");
    { int rcf = flush_state_ops(h); if (rcf) return rcf; }
    const size_t bytes = sizeof(State18) + sizeof(LioCtrl) + sizeof(VioCtrl) + sizeof(GridBarrier);
    FLB_CUDA(h, h->pin_res[slot].reserve(bytes));
    if (!h->ev_res[slot]) FLB_CUDA(h, cudaEventCreateWithFlags(&h->ev_res[slot], cudaEventDisableTiming));
    char* po = static_cast<char*>(h->pin_res[slot].p);
    {
        static_assert(sizeof(State18) % 4 == 0 && sizeof(LioCtrl) % 4 == 0 && sizeof(VioCtrl) % 4 == 0 && sizeof(GridBarrier) % 4 == 0, "word copies");
        void* dout = nullptr;
        FLB_CUDA(h, cudaHostGetDevicePointer(&dout, po, 0));
        LaunchScope ls(h, FAM_OTHER);
        k_pack_result<<<1, 256, 0, h->stream>>>(&h->states.p[0], reinterpret_cast<const unsigned*>(h->lio_ctrl.p), (int)(sizeof(LioCtrl) / 4),
                                                reinterpret_cast<const unsigned*>(h->vio_ctrl.p), (int)(sizeof(VioCtrl) / 4),
                                                reinterpret_cast<const unsigned*>(h->barrier.p), (int)(sizeof(GridBarrier) / 4),
                                                static_cast<unsigned*>(dout));
        FLB_CUDA(h, cudaGetLastError());
    }
    FLB_CUDA(h, cudaEventRecord(h->ev_res[slot], h->stream));
    h->res_pending[slot] = true;
    return FLB_OK;
}

int flb_state_download_wait(flb_handle* h, int slot, flb_state18* x, flb_lio_report* lio, flb_vio_report* vio) {
    FLB_CHECK_H(h);
    if (slot < 0 || slot > 1 || !h->res_pending[slot]) return fail(h, FLB_ERR_STATE, "flb_state_download_wait: nothing enqueued in this slot");
    FLB_CUDA(h, cudaEventSynchronize(h->ev_res[slot]));
    h->res_pending[slot] = false;
    const char* po = static_cast<const char*>(h->pin_res[slot].p);
    GridBarrier b;
    std::memcpy(&b, po + sizeof(State18) + sizeof(LioCtrl) + sizeof(VioCtrl), sizeof(b));
    if (b.timeout) {
        cudaMemset(h->barrier.p, 0, sizeof(GridBarrier));
        return fail(h, FLB_ERR_TIMEOUT, "device-side grid barrier watchdog tripped");
    }
    if (x) std::memcpy(x, po, sizeof(State18));
    if (lio) { LioCtrl c; std::memcpy(&c, po + sizeof(State18), sizeof(c)); fill_lio_report(c, lio); }
    if (vio) { VioCtrl c; std::memcpy(&c, po + sizeof(State18) + sizeof(LioCtrl), sizeof(c)); fill_vio_report(c, vio); }
    return FLB_OK;
}

int flb_lio_update_enqueue(flb_handle* h, const flb_lio_params* prm) {
    FLB_CHECK_H(h);
    if (!prm) return fail(h, FLB_ERR_INVALID, "null params");
    return enqueue_lio_update(h, prm);
}

int flb_vio_update_enqueue(flb_handle* h, const flb_vio_params* prm) {
    FLB_CHECK_H(h);
    if (!prm) return fail(h, FLB_ERR_INVALID, "null params");
    return enqueue_vio_update(h, prm);
}

// One frame in one call: uploads + both updates enqueued + (optionally) the pipelined read-back.
int flb_frame_enqueue(flb_handle* h, const flb_frame_inputs* in, const flb_lio_params* lprm, const flb_vio_params* vprm, int result_slot) {
    FLB_CHECK_H(h);
    if (!in || !lprm || !in->x || !in->x_prop) return fail(h, FLB_ERR_INVALID, "flb_frame_enqueue: null argument");
    int rc = flb_scan_upload(h, in->scan_xyz, in->n_scan, in->scan_stride);
    if (rc) return rc;
    rc = flb_state_upload(h, in->x, in->x_prop);
    if (rc) return rc;
    rc = enqueue_lio_update(h, lprm);
    if (rc) return rc;
    if (vprm) {
        if (in->gray) { rc = flb_image_upload(h, in->gray, in->width, in->height, in->stride_bytes); if (rc) return rc; }
        if (in->patch_pos) { rc = flb_patches_upload(h, in->patch_pos, in->patch, in->search_level, in->Pn); if (rc) return rc; }
        rc = flb_state_set_prior_enqueue(h);          // state_propagat = state (src/laserMapping.cpp:1292), zero-motion propagation
        if (rc) return rc;
        rc = enqueue_vio_update(h, vprm);
        if (rc) return rc;
    }
    if (result_slot >= 0) return flb_state_download_enqueue(h, result_slot);
    return FLB_OK;
}

int flb_lio_update(flb_handle* h, const flb_lio_params* prm, flb_state18* x, const flb_state18* x_prop, flb_lio_report* rep) {
    FLB_CHECK_H(h);
    if (!prm || !x || !x_prop) return fail(h, FLB_ERR_INVALID, "flb_lio_update: null argument");
    int rc = flb_state_upload(h, x, x_prop);
    if (rc) return rc;
    rc = enqueue_lio_update(h, prm);
    if (rc) return rc;
    flb_lio_report r{};
    rc = flb_state_download(h, x, &r, nullptr);
    if (rc) return rc;
    if (rep) *rep = r;
    if (r.status != 0) return fail(h, r.status, "flb_lio_update: device reported status %d (singular normal matrix?)", r.status);
    return FLB_OK;
}

// ---------------------------------------------------------------------------------------
int flb_lio_update_ikfom(flb_handle* h, const flb_ikfom_params* prm, flb_state_ikfom* x, flb_ikfom_report* rep) {
    FLB_CHECK_H(h);
    if (!prm || !x) return fail(h, FLB_ERR_INVALID, "flb_lio_update_ikfom: null argument");
    if (prm->max_iteration < 0) return fail(h, FLB_ERR_INVALID, "max_iteration < 0");
    if (h->M <= 0 || h->N <= 0) return fail(h, FLB_ERR_STATE, "flb_lio_update_ikfom: map and scan must be uploaded first");
    if (h->comm || h->p2p.world > 1) return fail(h, FLB_ERR_STATE, "flb_lio_update_ikfom: single-GPU only");
    void* stv = nullptr;
    FLB_CUDA(h, h->st_state.acquire(sizeof(StateIkfom), &stv));
    std::memcpy(stv, x, sizeof(StateIkfom));
    FLB_CUDA(h, cudaMemcpyAsync(&h->ik_states.p[0], stv, sizeof(StateIkfom), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, h->st_state.mark(h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(&h->ik_states.p[1], &h->ik_states.p[0], sizeof(StateIkfom), cudaMemcpyDeviceToDevice, h->stream));
    LioParamsDev d{};            // the extrinsic comes from the state every pass; only plane_thr / grid matter here
    LioArgs a = make_lio_args(h, d, false, 12);
    IkfomSolveArgs s{};
    s.state = &h->ik_states.p[0];
    s.state_prop = &h->ik_states.p[1];
    s.ctrl = h->ik_ctrl.p;
    s.prm.R = prm->laser_point_cov;
    s.prm.max_iteration = prm->max_iteration;
    std::memcpy(s.prm.limit, prm->limit, sizeof(s.prm.limit));
    const int cap = std::max(1, h->occ_ik * h->num_sms);
    const int want = std::min(cap, std::max(h->num_sms, std::min(2, h->occ_ik) * h->num_sms));
    const int grid = std::max(1, std::min((h->N + 31) / 32, want));
    FLB_CUDA(h, h->partials.reserve(std::max<size_t>((size_t)grid * lio_packed(12), h->partials.cap)));
    a.partials = h->partials.p;
    s.partials = h->partials.p;
    s.nblocks = grid;
    GridBarrier* bar = h->barrier.p;
    void* args[] = {&a, &s, &bar};
    {
        LaunchScope ls(h, FAM_LIO_KNN);
        FLB_CUDA(h, cudaLaunchCooperativeKernel((void*)k_lio_update_ikfom_persistent<kLioBlock>, dim3(grid), dim3(kLioBlock), args, 0,
                                                h->stream));
    }
    h->last_pass_valid = false;
    FLB_CUDA(h, h->pin_out.reserve(sizeof(StateIkfom) + sizeof(IkfomCtrl) + sizeof(GridBarrier)));
    char* po = static_cast<char*>(h->pin_out.p);
    FLB_CUDA(h, cudaMemcpyAsync(po, &h->ik_states.p[0], sizeof(StateIkfom), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(po + sizeof(StateIkfom), h->ik_ctrl.p, sizeof(IkfomCtrl), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(po + sizeof(StateIkfom) + sizeof(IkfomCtrl), h->barrier.p, sizeof(GridBarrier), cudaMemcpyDeviceToHost,
                                h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    GridBarrier b;
    std::memcpy(&b, po + sizeof(StateIkfom) + sizeof(IkfomCtrl), sizeof(b));
    if (b.timeout) {
        cudaMemset(h->barrier.p, 0, sizeof(GridBarrier));
        return fail(h, FLB_ERR_TIMEOUT, "device-side grid barrier watchdog tripped");
    }
    std::memcpy(x, po, sizeof(StateIkfom));
    IkfomCtrl c;
    std::memcpy(&c, po + sizeof(StateIkfom), sizeof(c));
    if (rep) {
        rep->passes = c.passes; rep->knn_passes = c.knn_passes; rep->n_eff_last = c.n_eff_last;
        rep->converged_last = c.converged_last; rep->res_mean_last = c.res_mean_last; rep->rows_total = c.rows_total;
        rep->status = c.status;
    }
    if (c.status != 0) return fail(h, c.status, "flb_lio_update_ikfom: device reported status %d", c.status);
    return FLB_OK;
}

// ---------------------------------------------------------------------------------------
int flb_image_upload(flb_handle* h, const uint8_t* gray, int width, int height, int stride) {
    FLB_CHECK_H(h);
    if (!gray || width < 16 || height < 16 || stride < width) return fail(h, FLB_ERR_INVALID, "flb_image_upload: bad arguments");
    FLB_CUDA(h, h->img_alt.reserve((size_t)width * height));
    const unsigned char* src = gray;
    const bool direct = (stride == width) && is_pinned(gray);     // page-locked caller buffer: no staging copy
    if (!direct) {
        void* stv = nullptr;
        FLB_CUDA(h, h->st_img.acquire((size_t)width * height, &stv));
        unsigned char* st = static_cast<unsigned char*>(stv);
        if (stride == width) std::memcpy(st, gray, (size_t)width * height);
        else for (int r = 0; r < height; ++r) std::memcpy(st + (size_t)r * width, gray + (size_t)r * stride, width);
        src = st;
    }
    { int rcq = vio_copy_begin(h, h->img_slot); if (rcq) return rcq; }
    FLB_CUDA(h, cudaMemcpyAsync(h->img_alt.p, src, (size_t)width * height, cudaMemcpyHostToDevice, h->copy_stream));
    if (!direct) FLB_CUDA(h, h->st_img.mark(h->copy_stream));
    { int rcq = vio_copy_end(h); if (rcq) return rcq; }
    std::swap(h->img, h->img_alt);
    h->img_slot.slot ^= 1;
    h->img_w = width;
    h->img_h = height;
    h->last_vio_valid = false;
    return FLB_OK;
}

int flb_patches_upload(flb_handle* h, const double* pos, const float* patch, const int* search_level, int Pn) {
    FLB_CHECK_H(h);
    if (Pn < 0 || (Pn > 0 && (!pos || !patch || !search_level))) return fail(h, FLB_ERR_INVALID, "flb_patches_upload: bad arguments");
    for (int i = 0; i < Pn; ++i)
        if (search_level[i] < 0 || search_level[i] > 2) return fail(h, FLB_ERR_INVALID, "search_level[%d] = %d outside [0,2]", i, search_level[i]);
    const size_t n = (size_t)std::max(Pn, 1);
    FLB_CUDA(h, h->patch_pos_alt.reserve(n * 3));
    FLB_CUDA(h, h->patch_ref_alt.reserve(n * 192));
    FLB_CUDA(h, h->patch_level_alt.reserve(n));
    FLB_CUDA(h, h->errors.reserve(2 * n));
    h->err_stride = (int)n;
    const int nb = (Pn + 7) / 8;
    FLB_CUDA(h, h->partials.reserve(std::max<size_t>((size_t)std::max(nb, 1) * kVioPacked, h->partials.cap)));
    const size_t bytes = n * (3 * sizeof(double) + 192 * sizeof(float) + sizeof(int)) + 16;
    if (Pn > 0) {
        const bool direct = is_pinned(pos) && is_pinned(patch) && is_pinned(search_level);
        { int rcq = vio_copy_begin(h, h->patch_slot); if (rcq) return rcq; }
        if (direct) {
            FLB_CUDA(h, cudaMemcpyAsync(h->patch_pos_alt.p, pos, (size_t)Pn * 3 * sizeof(double), cudaMemcpyHostToDevice, h->copy_stream));
            FLB_CUDA(h, cudaMemcpyAsync(h->patch_ref_alt.p, patch, (size_t)Pn * 192 * sizeof(float), cudaMemcpyHostToDevice, h->copy_stream));
            FLB_CUDA(h, cudaMemcpyAsync(h->patch_level_alt.p, search_level, (size_t)Pn * sizeof(int), cudaMemcpyHostToDevice, h->copy_stream));
        } else {
            // pageable caller buffers: pack into pinned staging and hand each piece to the copy engine as soon
            // as it is packed, the reference patches (96 % of the bytes) in four slices, so that the transfer
            // runs behind the host memcpy instead of after it
            void* stv = nullptr;
            FLB_CUDA(h, h->st_patch.acquire(bytes, &stv));
            char* b = static_cast<char*>(stv);
            std::memcpy(b, pos, (size_t)Pn * 3 * sizeof(double));
            FLB_CUDA(h, cudaMemcpyAsync(h->patch_pos_alt.p, b, (size_t)Pn * 3 * sizeof(double), cudaMemcpyHostToDevice, h->copy_stream));
            char* b3 = b + (size_t)Pn * 3 * sizeof(double);
            std::memcpy(b3, search_level, (size_t)Pn * sizeof(int));
            FLB_CUDA(h, cudaMemcpyAsync(h->patch_level_alt.p, b3, (size_t)Pn * sizeof(int), cudaMemcpyHostToDevice, h->copy_stream));
            char* b2 = b3 + (((size_t)Pn * sizeof(int) + 15) & ~(size_t)15);
            const size_t total = (size_t)Pn * 192, slice = (total + 3) / 4;
            for (size_t o = 0; o < total; o += slice) {
                const size_t cnt = std::min(slice, total - o);
                std::memcpy(b2 + o * sizeof(float), patch + o, cnt * sizeof(float));
                FLB_CUDA(h, cudaMemcpyAsync(h->patch_ref_alt.p + o, b2 + o * sizeof(float), cnt * sizeof(float), cudaMemcpyHostToDevice, h->copy_stream));
            }
        }
        if (!direct) FLB_CUDA(h, h->st_patch.mark(h->copy_stream));
        { int rcq = vio_copy_end(h); if (rcq) return rcq; }
    }
    std::swap(h->patch_pos, h->patch_pos_alt);
    std::swap(h->patch_ref, h->patch_ref_alt);
    std::swap(h->patch_level, h->patch_level_alt);
    h->patch_slot.slot ^= 1;
    if (h->comm) {
        // agree on the largest shard so every rank contributes an equal-size block to ncclAllGather;
        // the padding entries stay 0.0f, and adding 0.0f to the sequential float sum is exact.
        int* dmax = reinterpret_cast<int*>(h->packed.p);
        FLB_CUDA(h, cudaMemcpyAsync(dmax, &Pn, sizeof(int), cudaMemcpyHostToDevice, h->stream));
        int r = g_nccl.AllReduce(dmax, dmax, 1, kNcclInt32, kNcclMax, h->comm, h->stream);
        if (r != 0) return fail(h, FLB_ERR_COMM, "ncclAllReduce(max Pn) failed");
        int shard = 0;
        FLB_CUDA(h, cudaMemcpyAsync(&shard, dmax, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        FLB_CUDA(h, cudaStreamSynchronize(h->stream));
        h->err_shard = std::max(shard, 1);
        h->err_stride = std::max(h->err_stride, h->err_shard);
        FLB_CUDA(h, h->errors.reserve(2 * (size_t)h->err_stride));
        FLB_CUDA(h, h->errors_all.reserve((size_t)h->err_shard * (size_t)h->world));
    }
    FLB_CUDA(h, cudaMemsetAsync(h->errors.p, 0, h->errors.cap * sizeof(float), h->stream));
    h->Pn = Pn;
    h->pn_on_device = false;
    h->last_vio_valid = false;
    return FLB_OK;
}

int flb_camera_set(flb_handle* h, const flb_camera* cam) {
    FLB_CHECK_H(h);
    if (!cam || cam->width < 16 || cam->height < 16 || !(std::fabs(cam->fx) > 0) || !(std::fabs(cam->fy) > 0))
        return fail(h, FLB_ERR_INVALID, "flb_camera_set: bad camera");
    CamModel c{};
    c.width = cam->width;
    c.height = cam->height;
    c.fx = cam->fx; c.fy = cam->fy; c.cx = cam->cx; c.cy = cam->cy;
    for (int i = 0; i < 5; ++i) c.d[i] = cam->d[i];
    // vikit PinholeCamera::errorMultiplier2() = |fx|, errorMultiplier() = |4 fx fy| (src/lidar_selection.cpp:58-59)
    c.jfx = std::fabs(cam->fx);
    c.jfy = std::fabs(4.0 * cam->fx * cam->fy) / (4. * c.jfx);
    h->cam = c;
    h->cam_set = true;
    return FLB_OK;
}

int flb_vio_pass(flb_handle* h, const flb_vio_params* prm, const double R[9], const double p[3], int level, flb_vio_eq* out) {
    FLB_CHECK_H(h);
    if (!prm || !R || !p || !out || level < 0 || level > 2) return fail(h, FLB_ERR_INVALID, "flb_vio_pass: bad arguments");
    if (!h->cam_set || h->img_w <= 0) return fail(h, FLB_ERR_STATE, "flb_vio_pass: camera and image must be set first");
    if (h->cam.width != h->img_w || h->cam.height != h->img_h) return fail(h, FLB_ERR_STATE, "camera / image size mismatch");
    std::memset(out, 0, sizeof(*out));
    { int rcp = resolve_pn(h); if (rcp) return rcp; }
    if (h->Pn == 0) return FLB_OK;
    { int rcq = vio_inputs_acquire(h); if (rcq) return rcq; }
    const size_t Pn = h->Pn;
    FLB_CUDA(h, h->x_z.reserve(Pn * 64));
    FLB_CUDA(h, h->x_H.reserve(Pn * 64 * 6));
    VioParamsDev d;
    to_dev_params(prm, d);
    void* stv = nullptr;
    FLB_CUDA(h, h->st_misc.acquire(12 * sizeof(double), &stv));
    double* st = static_cast<double*>(stv);
    std::memcpy(st, R, 9 * sizeof(double));
    std::memcpy(st + 9, p, 3 * sizeof(double));
    FLB_CUDA(h, cudaMemcpyAsync(h->pose12.p, st, 12 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, h->st_misc.mark(h->stream));
    VioArgs a{};
    a.img = h->img.p;
    a.cam = h->cam;
    a.pos = h->patch_pos.p;
    a.patch = h->patch_ref.p;
    a.search_level = h->patch_level.p;
    a.Pn = h->Pn;
    a.state = &h->states.p[0];
    a.pose_override = h->pose12.p;
    a.prm = d;
    a.ctrl = h->vio_ctrl.p;
    a.force_level = level;
    a.errors = h->errors.p;
    a.err_stride = h->err_stride;
    a.partials = h->partials.p;
    a.x_z = h->x_z.p;
    a.x_H = h->x_H.p;
    const int nb = vio_nblocks(h);
    {
        LaunchScope ls(h, FAM_VIO);
        k_vio_pass<kVioBlock><<<nb, kVioBlock, 0, h->stream>>>(a);
        FLB_CUDA(h, cudaGetLastError());
    }
    {
        LaunchScope ls(h, FAM_SOLVE);
        k_reduce_only<<<1, 32, 0, h->stream>>>(h->partials.p, nb, kVioPacked, h->packed.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    { int rcq = vio_inputs_release(h); if (rcq) return rcq; }
    FLB_CUDA(h, h->pin_out.reserve(kVioPacked * sizeof(double) + Pn * sizeof(float)));
    double* po = static_cast<double*>(h->pin_out.p);
    float* pe = reinterpret_cast<float*>(po + kVioPacked);
    FLB_CUDA(h, cudaMemcpyAsync(po, h->packed.p, kVioPacked * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(pe, h->errors.p, Pn * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    int k = 0;
    for (int r = 0; r < 6; ++r)
        for (int c = r; c < 6; ++c) {
            out->HTH[r * 6 + c] = po[k];
            out->HTH[c * 6 + r] = po[k];
            ++k;
        }
    for (int r = 0; r < 6; ++r) out->HTz[r] = po[21 + r];
    out->n_meas = (int64_t)po[27];
    out->skipped = (int)po[28];
    // error = sum_i errors[i] (float, patch order) / n_meas  (src/lidar_selection.cpp:852,857)
    float e = 0.0f;
    for (size_t i = 0; i < Pn; ++i) e = e + pe[i];
    out->error = e / (float)(size_t)out->n_meas;
    h->last_vio_valid = true;
    return FLB_OK;
}

int flb_vio_export(flb_handle* h, double* z, double* H_sub, float* errors) {
    FLB_CHECK_H(h);
    if (!h->last_vio_valid) return fail(h, FLB_ERR_STATE, "flb_vio_export: no flb_vio_pass to export");
    const size_t Pn = h->Pn;
    if (z) FLB_CUDA(h, cudaMemcpyAsync(z, h->x_z.p, Pn * 64 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (H_sub) FLB_CUDA(h, cudaMemcpyAsync(H_sub, h->x_H.p, Pn * 64 * 6 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (errors) FLB_CUDA(h, cudaMemcpyAsync(errors, h->errors.p, Pn * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    return FLB_OK;
}

int flb_vio_errors(flb_handle* h, float* errors, int capacity) {
    FLB_CHECK_H(h);
    if (!errors || capacity < 0) return fail(h, FLB_ERR_INVALID, "flb_vio_errors: bad arguments");
    { int rcp = resolve_pn(h); if (rcp) return rcp; }
    const int n = std::min(capacity, h->Pn);
    if (n == 0) return FLB_OK;
    // which half the last executed pass of the last update wrote is part of the device control block
    VioCtrl c;
    FLB_CUDA(h, cudaMemcpyAsync(&c, h->vio_ctrl.p, sizeof(VioCtrl), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    const int buf = (c.err_buf == 1) ? 1 : 0;
    FLB_CUDA(h, cudaMemcpyAsync(errors, h->errors.p + (size_t)buf * h->err_stride, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    return FLB_OK;
}

int flb_vio_update_level(flb_handle* h, const flb_vio_params* prm, int level, float total_residual, flb_state18* x,
                         const flb_state18* x_prop, float* last_error, double* G18x6, flb_vio_report* rep) {
    FLB_CHECK_H(h);
    if (!prm || !x || !x_prop || level < 0 || level > 2) return fail(h, FLB_ERR_INVALID, "flb_vio_update_level: bad arguments");
    if (!h->cam_set || h->img_w <= 0) return fail(h, FLB_ERR_STATE, "flb_vio_update_level: camera and image must be set first");
    if (h->cam.width != h->img_w || h->cam.height != h->img_h) return fail(h, FLB_ERR_STATE, "camera / image size mismatch");
    if (h->comm || h->p2p.world > 1) return fail(h, FLB_ERR_STATE, "flb_vio_update_level: single GPU");
    { int rcp = resolve_pn(h); if (rcp) return rcp; }
    if (last_error) *last_error = 0.f;                               // :746 (total_points == 0 returns 0.)
    flb_vio_report r{};
    if (h->Pn == 0) { if (rep) *rep = r; return FLB_OK; }
    int rc = flb_state_upload(h, x, x_prop);
    if (rc) return rc;
    VioParamsDev d;
    to_dev_params(prm, d);
    d.single_level = 1;
    { int rcq = vio_inputs_acquire(h); if (rcq) return rcq; }
    VioSolveArgs s{};
    s.state = &h->states.p[0];
    s.state_prop = &h->states.p[1];
    s.old_state = &h->states.p[2];
    s.ctrl = h->vio_ctrl.p;
    s.prior = h->prior.p;
    s.G_last = h->G_last.p;
    s.partials = h->partials.p;
    s.nblocks = vio_nblocks(h);
    s.errors = h->errors.p;
    s.err_stride = h->err_stride;
    s.Pn_total = h->Pn;
    s.prm = d;
    s.timeout_flag = &h->barrier.p->timeout;
    VioArgs a{};
    a.img = h->img.p;
    a.cam = h->cam;
    a.pos = h->patch_pos.p;
    a.patch = h->patch_ref.p;
    a.search_level = h->patch_level.p;
    a.Pn = h->Pn;
    a.state = &h->states.p[0];
    a.prm = d;
    a.ctrl = h->vio_ctrl.p;
    a.force_level = -1;
    a.errors = h->errors.p;
    a.err_stride = h->err_stride;
    a.partials = h->partials.p;
    {
        LaunchScope ls(h, FAM_SOLVE);
        k_vio_begin_level<<<1, 32, 0, h->stream>>>(h->vio_ctrl.p, h->Pn, level, total_residual);
        FLB_CUDA(h, cudaGetLastError());
    }
    const int nb = vio_nblocks(h);
    for (int it = 0; it < std::max(prm->max_iteration, 0); ++it) {      // later launches return at once when the level has ended
        {
            LaunchScope ls(h, FAM_VIO);
            k_vio_pass<kVioBlock><<<nb, kVioBlock, 0, h->stream>>>(a);
            FLB_CUDA(h, cudaGetLastError());
        }
        LaunchScope ls(h, FAM_SOLVE);
        k_vio_finalize<<<1, kLeaderBlock, 0, h->stream>>>(s);
        FLB_CUDA(h, cudaGetLastError());
    }
    if (G18x6) {
        LaunchScope ls(h, FAM_SOLVE);
        k_vio_export_gain<<<1, kLeaderBlock, 0, h->stream>>>(s, h->packed.p);
        FLB_CUDA(h, cudaGetLastError());
        FLB_CUDA(h, cudaMemcpyAsync(G18x6, h->packed.p, 108 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    }
    { int rcq = vio_inputs_release(h); if (rcq) return rcq; }
    h->last_vio_valid = false;
    rc = flb_state_download(h, x, nullptr, &r);
    if (rc) return rc;
    if (rep) *rep = r;
    if (last_error) *last_error = r.last_error[level];               // return last_error (:901)
    if (r.status != 0) return fail(h, r.status, "flb_vio_update_level: device reported status %d", r.status);
    return FLB_OK;
}

int flb_vio_update(flb_handle* h, const flb_vio_params* prm, flb_state18* x, const flb_state18* x_prop, flb_vio_report* rep) {
    FLB_CHECK_H(h);
    if (!prm || !x || !x_prop) return fail(h, FLB_ERR_INVALID, "flb_vio_update: null argument");
    if (h->cam_set && (h->cam.width != h->img_w || h->cam.height != h->img_h))
        return fail(h, FLB_ERR_STATE, "camera / image size mismatch");
    int rc = flb_state_upload(h, x, x_prop);
    if (rc) return rc;
    rc = enqueue_vio_update(h, prm);
    if (rc) return rc;
    flb_vio_report r{};
    rc = flb_state_download(h, x, nullptr, &r);
    if (rc) return rc;
    if (rep) *rep = r;
    if (r.status != 0) return fail(h, r.status, "flb_vio_update: device reported status %d", r.status);
    return FLB_OK;
}

// ---------------------------------------------------------------------------------------
int flb_profile_start(flb_handle* h) {
    FLB_CHECK_H(h);
    for (auto& ev : h->evs) { cudaEventDestroy(ev.a); cudaEventDestroy(ev.b); }
    h->evs.clear();
    h->profiling = true;
    return FLB_OK;
}

int flb_profile_stop(flb_handle* h, double ms[4], int64_t launches[4]) {
    FLB_CHECK_H(h);
    h->profiling = false;
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    for (int i = 0; i < 4; ++i) { if (ms) ms[i] = 0.0; if (launches) launches[i] = 0; }
    for (auto& ev : h->evs) {
        float t = 0.f;
        cudaEventElapsedTime(&t, ev.a, ev.b);
        if (ev.fam < 4) {
            if (ms) ms[ev.fam] += t;
            if (launches) launches[ev.fam] += 1;
        }
        cudaEventDestroy(ev.a);
        cudaEventDestroy(ev.b);
    }
    h->evs.clear();
    return FLB_OK;
}

int flb_trace_enable(flb_handle* h, int on) {
    FLB_CHECK_H(h);
    h->tracing = on != 0;
    FLB_CUDA(h, cudaMemsetAsync(h->trace.p, 0, 2 * kTraceLen * sizeof(unsigned long long), h->stream));
    return FLB_OK;
}

// Test aid (not part of the public header): move the pose-packet flag base, e.g. next to its wrap-around point
// (the base advances by 4096 per persistent launch and is re-based, with the packet cleared, before it overflows).
int flb_debug_set_packet_epoch(flb_handle* h, unsigned epoch) {
    FLB_CHECK_H(h);
    h->pkt_epoch = epoch;
    return FLB_OK;
}

// Tracing aid (not part of the public header): per-block / per-warp stamps of the last VIO pass,
// kVioDbg words per block.
int flb_debug_vio_stamps(flb_handle* h, unsigned long long* out, int max_blocks, int* nblocks, int* words_per_block) {
    FLB_CHECK_H(h);
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    const int n = std::min(h->dbg_vio_blocks, max_blocks);
    if (n > 0) FLB_CUDA(h, cudaMemcpy(out, h->dbg_vio.p, (size_t)n * kVioDbg * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    *nblocks = n;
    *words_per_block = kVioDbg;
    return FLB_OK;
}

// Test aid: force the scan ordering path of the following uploads (0 automatic, 1 one-block kernel, 2 device-wide sort).
int flb_debug_set_scan_sort(flb_handle* h, int mode) {
    FLB_CHECK_H(h);
    if (mode < 0 || mode > 2) return fail(h, FLB_ERR_INVALID, "flb_debug_set_scan_sort: mode 0, 1 or 2");
    h->scan_sort_mode = mode;
    return FLB_OK;
}

// Test aid: the uploaded scan's order -- src_index[i] = index (in the caller's array) of the point at sorted position i.
int flb_debug_scan_order(flb_handle* h, int* src_index, int capacity) {
    FLB_CHECK_H(h);
    if (!src_index || capacity < h->N) return fail(h, FLB_ERR_INVALID, "flb_debug_scan_order: bad arguments");
    if (h->N == 0) return FLB_OK;
    std::vector<float4> tmp((size_t)h->N);
    FLB_CUDA(h, cudaMemcpyAsync(tmp.data(), h->scan.p, (size_t)h->N * sizeof(float4), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    for (int i = 0; i < h->N; ++i) std::memcpy(&src_index[i], &tmp[(size_t)i].w, sizeof(int));
    return FLB_OK;
}

int flb_debug_block_stamps(flb_handle* h, unsigned long long* out, int max_blocks, int* nblocks) {
    FLB_CHECK_H(h);
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    const int n = std::min(h->dbg_blocks, max_blocks);     // 16 words per block: 4 block stamps, 8 warp stamps
    if (n > 0) FLB_CUDA(h, cudaMemcpy(out, h->dbg.p, (size_t)n * 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    *nblocks = n;
    return FLB_OK;
}

int flb_trace_download(flb_handle* h, int which, double* us, int max_entries, int* n_entries) {
    FLB_CHECK_H(h);
    if (!us || !n_entries || (which != 0 && which != 1)) return fail(h, FLB_ERR_INVALID, "flb_trace_download: bad arguments");
    unsigned long long t[kTraceLen];
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    FLB_CUDA(h, cudaMemcpy(t, h->trace.p + which * kTraceLen, sizeof(t), cudaMemcpyDeviceToHost));
    int n = 0;
    for (int i = 1; i < kTraceLen && i - 1 < max_entries; ++i) {
        if (t[i] == 0 && i < 64) { if (max_entries < kTraceLen - 1) break; us[n++] = 0.0; continue; }
        us[n++] = t[i] ? (double)(t[i] - t[0]) * 1e-3 : 0.0;
    }
    *n_entries = n;
    return FLB_OK;
}

// ---------------------------------------------------------------------------------------
int flb_comm_unique_id(void* unique_id_128b) {
    if (!unique_id_128b) return FLB_ERR_INVALID;
    if (!g_nccl.load()) return fail(nullptr, FLB_ERR_COMM, "libnccl.so.2 not found");
    ncclUniqueId id;
    int r = g_nccl.GetUniqueId(&id);
    if (r != 0) return fail(nullptr, FLB_ERR_COMM, "ncclGetUniqueId failed (%d)", r);
    std::memcpy(unique_id_128b, &id, 128);
    return FLB_OK;
}

int flb_comm_init(flb_handle* h, const void* unique_id_128b, int rank, int world_size) {
    FLB_CHECK_H(h);
    if (!unique_id_128b || world_size < 1 || rank < 0 || rank >= world_size) return fail(h, FLB_ERR_INVALID, "flb_comm_init: bad arguments");
    if (!g_nccl.load()) return fail(h, FLB_ERR_COMM, "libnccl.so.2 not found");
    if (h->comm) { g_nccl.CommDestroy(h->comm); h->comm = nullptr; }
    ncclUniqueId id;
    std::memcpy(&id, unique_id_128b, 128);
    int r = g_nccl.CommInitRank(&h->comm, world_size, id, rank);
    if (r != 0) { h->comm = nullptr; return fail(h, FLB_ERR_COMM, "ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"); }
    h->rank = rank;
    h->world = world_size;
    return FLB_OK;
}

// ---- fused NVLink exchange -------------------------------------------------------------------
int flb_p2p_export(flb_handle* h, void* handle_64b) {
    FLB_CHECK_H(h);
    if (!handle_64b) return fail(h, FLB_ERR_INVALID, "flb_p2p_export: null handle buffer");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    FLB_CUDA(h, h->mailbox.reserve(1));
    FLB_CUDA(h, h->p2p_seq.reserve(1));
    FLB_CUDA(h, cudaMemset(h->mailbox.p, 0, sizeof(P2PMailbox)));
    FLB_CUDA(h, cudaMemset(h->p2p_seq.p, 0, sizeof(unsigned long long)));
    cudaIpcMemHandle_t ih;
    FLB_CUDA(h, cudaIpcGetMemHandle(&ih, h->mailbox.p));
    std::memcpy(handle_64b, &ih, 64);
    return FLB_OK;
}

int flb_p2p_attach(flb_handle* h, int rank, int world_size, const void* handles) {
    FLB_CHECK_H(h);
    if (!handles || world_size < 1 || world_size > kP2PMaxWorld || rank < 0 || rank >= world_size)
        return fail(h, FLB_ERR_INVALID, "flb_p2p_attach: bad arguments (world <= %d)", kP2PMaxWorld);
    if (!h->mailbox.p) return fail(h, FLB_ERR_STATE, "flb_p2p_attach: call flb_p2p_export first");
    P2PArgs a{};
    a.world = world_size;
    a.rank = rank;
    a.seq = h->p2p_seq.p;
    for (int r = 0; r < world_size; ++r) {
        if (r == rank) { a.mail[r] = h->mailbox.p; continue; }
        cudaIpcMemHandle_t ih;
        std::memcpy(&ih, static_cast<const char*>(handles) + 64 * (size_t)r, 64);
        void* ptr = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&ptr, ih, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) return fail(h, FLB_ERR_COMM, "cudaIpcOpenMemHandle(rank %d): %s", r, cudaGetErrorString(e));
        h->p2p_peer_ptr[r] = ptr;
        a.mail[r] = static_cast<P2PMailbox*>(ptr);
    }
    h->p2p = a;
    h->rank = rank;
    h->world = world_size;
    return FLB_OK;
}

int flb_p2p_detach(flb_handle* h) {
    FLB_CHECK_H(h);
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    for (int r = 0; r < kP2PMaxWorld; ++r)
        if (h->p2p_peer_ptr[r]) { cudaIpcCloseMemHandle(h->p2p_peer_ptr[r]); h->p2p_peer_ptr[r] = nullptr; }
    h->p2p = P2PArgs{};
    return FLB_OK;
}

int flb_comm_destroy(flb_handle* h) {
    FLB_CHECK_H(h);
    if (h->comm) { g_nccl.CommDestroy(h->comm); h->comm = nullptr; }
    h->world = 1;
    h->rank = 0;
    return FLB_OK;
}

}  // extern "C"

// =======================================================================================
// Batched frames (SURVEY.md section 7 H2(iv)): B independent frames per launch
// =======================================================================================
extern "C" {

int flb_batch_begin(flb_handle* h, int B, int max_points_per_frame) {
    FLB_CHECK_H(h);
    if (B < 1 || B > 4096 || max_points_per_frame < 1) return fail(h, FLB_ERR_INVALID, "flb_batch_begin: bad arguments");
    if (h->M <= 0) return fail(h, FLB_ERR_STATE, "flb_batch_begin: upload the map first");
    auto& b = h->batch;
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    b.B = B;
    b.n_cap = (max_points_per_frame + kLioBlock - 1) / kLioBlock * kLioBlock;
    b.N.assign(B, 0);
    const size_t tot = (size_t)B * b.n_cap;
    FLB_CUDA(h, b.scan.reserve(tot));
    FLB_CUDA(h, b.plane.reserve(tot));
    FLB_CUDA(h, b.sel.reserve(tot));
    FLB_CUDA(h, b.plane_ok.reserve(tot));
    FLB_CUDA(h, b.states.reserve((size_t)B * 5));
    FLB_CUDA(h, b.lio_ctrl.reserve(B));
    FLB_CUDA(h, b.vio_ctrl.reserve(B));
    FLB_CUDA(h, b.prior.reserve(B));
    FLB_CUDA(h, b.G_last.reserve((size_t)B * 108));
    FLB_CUDA(h, b.lio_args.reserve(B));
    FLB_CUDA(h, b.lio_solve.reserve(B));
    FLB_CUDA(h, b.vio_args.reserve(B));
    FLB_CUDA(h, b.vio_solve.reserve(B));
    FLB_CUDA(h, b.lio_ctrl_ptrs.reserve(B));
    FLB_CUDA(h, b.vio_ctrl_ptrs.reserve(B));
    std::vector<LioCtrl*> lp(B);
    std::vector<VioCtrl*> vp(B);
    for (int i = 0; i < B; ++i) { lp[i] = b.lio_ctrl.p + i; vp[i] = b.vio_ctrl.p + i; }
    FLB_CUDA(h, cudaMemcpy(b.lio_ctrl_ptrs.p, lp.data(), B * sizeof(LioCtrl*), cudaMemcpyHostToDevice));
    FLB_CUDA(h, cudaMemcpy(b.vio_ctrl_ptrs.p, vp.data(), B * sizeof(VioCtrl*), cudaMemcpyHostToDevice));
    FLB_CUDA(h, cudaMemset(b.lio_ctrl.p, 0, B * sizeof(LioCtrl)));
    FLB_CUDA(h, cudaMemset(b.vio_ctrl.p, 0, B * sizeof(VioCtrl)));
    return FLB_OK;
}

int flb_batch_set_frame(flb_handle* h, int frame, const float* body_xyz, int N, int stride, const flb_state18* x, const flb_state18* x_prop) {
    FLB_CHECK_H(h);
    auto& b = h->batch;
    if (frame < 0 || frame >= b.B || !x || !x_prop || N < 1 || N > b.n_cap) return fail(h, FLB_ERR_INVALID, "flb_batch_set_frame: bad arguments");
    int rc = flb_scan_upload(h, body_xyz, N, stride);      // validates, Morton-sorts into h->scan
    if (rc) return rc;
    const size_t off = (size_t)frame * b.n_cap;
    FLB_CUDA(h, cudaMemcpyAsync(b.scan.p + off, h->scan.p, (size_t)N * sizeof(float4), cudaMemcpyDeviceToDevice, h->stream));
    FLB_CUDA(h, cudaMemsetAsync(b.sel.p + off, 1, N, h->stream));
    FLB_CUDA(h, cudaMemsetAsync(b.plane_ok.p + off, 0, N, h->stream));
    rc = flb_state_upload(h, x, x_prop);                   // through the handle's staging, then into the frame's slots
    if (rc) return rc;
    State18* st = b.states.p + (size_t)frame * 5;
    FLB_CUDA(h, cudaMemcpyAsync(st, &h->states.p[0], 2 * sizeof(State18), cudaMemcpyDeviceToDevice, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(st + 3, &h->states.p[0], 2 * sizeof(State18), cudaMemcpyDeviceToDevice, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    b.N[frame] = N;
    b.n_max = *std::max_element(b.N.begin(), b.N.end());
    return FLB_OK;
}

/* restore every frame's x / x_prop to what flb_batch_set_frame gave it (benchmark loop) */
int flb_batch_state_reset_enqueue(flb_handle* h) {
    FLB_CHECK_H(h);
    auto& b = h->batch;
    if (b.B < 1) return fail(h, FLB_ERR_STATE, "flb_batch_state_reset_enqueue: no batch");
    FLB_CUDA(h, cudaMemcpy2DAsync(b.states.p, 5 * sizeof(State18), b.states.p + 3, 5 * sizeof(State18), 2 * sizeof(State18), b.B,
                                  cudaMemcpyDeviceToDevice, h->stream));
    return FLB_OK;
}

int flb_batch_update_enqueue(flb_handle* h, const flb_lio_params* lprm, const flb_vio_params* vprm) {
    FLB_CHECK_H(h);
    auto& b = h->batch;
    if (b.B < 1 || b.n_max < 1) return fail(h, FLB_ERR_STATE, "flb_batch_update_enqueue: flb_batch_begin / flb_batch_set_frame first");
    if (!lprm) return fail(h, FLB_ERR_INVALID, "flb_batch_update_enqueue: null LIO params");
    if (h->comm || h->p2p.world > 1) return fail(h, FLB_ERR_STATE, "batched frames: single GPU");
    for (int i = 0; i < b.B; ++i)
        if (b.N[i] < 1) return fail(h, FLB_ERR_STATE, "flb_batch_update_enqueue: frame %d not set", i);
    const int B = b.B;
    const bool vio = vprm != nullptr && h->Pn > 0 && vprm->max_iteration > 0;
    if (vio) {
        if (!h->cam_set || h->img_w <= 0) return fail(h, FLB_ERR_STATE, "flb_batch_update_enqueue: camera and image must be set first");
        if (h->pn_on_device) { int rc = resolve_pn(h); if (rc) return rc; }
    }
    const int nb_lio = (b.n_max + kLioBlock - 1) / kLioBlock;
    const int nb_vio = (h->Pn + (kVioBlock / 32) - 1) / (kVioBlock / 32);
    b.partials_per = (size_t)std::max(nb_lio * lio_packed(6), nb_vio * kVioPacked);
    FLB_CUDA(h, b.partials.reserve((size_t)B * b.partials_per));
    const int estride = std::max(h->Pn, 1);
    FLB_CUDA(h, b.errors.reserve((size_t)B * 2 * estride));
    LioParamsDev ld;
    to_dev_params(lprm, ld);
    std::vector<LioArgs> la(B);
    std::vector<LioSolveArgs> ls(B);
    for (int i = 0; i < B; ++i) {
        const size_t off = (size_t)i * b.n_cap;
        LioArgs a{};
        a.scan = b.scan.p + off;
        a.N = b.N[i];
        a.grid = h->grid;
        a.cell_start = h->cell_start.p;
        a.map_pts = h->map_pts.p;
        a.state = b.states.p + (size_t)i * 5;
        a.prm = ld;
        a.plane_thr = (float)h->cfg.plane_threshold;
        a.ctrl = b.lio_ctrl.p + i;
        a.force_rematch = -1;
        a.sel = b.sel.p + off;
        a.plane = b.plane.p + off;
        a.plane_ok = b.plane_ok.p + off;
        a.partials = b.partials.p + (size_t)i * b.partials_per;
        a.M = h->M;
        la[i] = a;
        LioSolveArgs s{};
        s.state = b.states.p + (size_t)i * 5;
        s.state_prop = s.state + 1;
        s.ctrl = b.lio_ctrl.p + i;
        s.prior = b.prior.p + i;
        s.partials = a.partials;
        s.nblocks = (b.N[i] + kLioBlock - 1) / kLioBlock;
        s.prm = ld;
        s.timeout_flag = &h->barrier.p->timeout;
        ls[i] = s;
    }
    // argument tables: pageable -> device through the stream (small; ordered before the launches that read them)
    FLB_CUDA(h, cudaMemcpyAsync(b.lio_args.p, la.data(), B * sizeof(LioArgs), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(b.lio_solve.p, ls.data(), B * sizeof(LioSolveArgs), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));          // la / ls are stack-owned
    {
        LaunchScope lsx(h, FAM_SOLVE);
        k_lio_begin_batched<<<(B + 127) / 128, 128, 0, h->stream>>>(b.lio_ctrl_ptrs.p, B);
        FLB_CUDA(h, cudaGetLastError());
    }
    const int T = lprm->max_iteration;
    for (int it = -1; it < T; ++it) {
        {
            // family tag: with early stop disabled the rematch passes are the first and the last (Appendix A)
            LaunchScope lsx(h, (it == -1 || it == T - 1) ? FAM_LIO_KNN : FAM_LIO_PLAIN);
            k_lio_pass_batched<6, kLioBlock><<<dim3(nb_lio, B), kLioBlock, 0, h->stream>>>(b.lio_args.p);
            FLB_CUDA(h, cudaGetLastError());
        }
        LaunchScope lsx(h, FAM_SOLVE);
        k_lio_finalize_batched<<<B, kLeaderBlock, 0, h->stream>>>(b.lio_solve.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    if (!vio) return FLB_OK;
    // state_propagat := the LIO posterior (zero-motion propagation between the two updates), per frame
    FLB_CUDA(h, cudaMemcpy2DAsync(b.states.p + 1, 5 * sizeof(State18), b.states.p, 5 * sizeof(State18), sizeof(State18), B,
                                  cudaMemcpyDeviceToDevice, h->stream));
    { int rcq = vio_inputs_acquire(h); if (rcq) return rcq; }
    VioParamsDev vd;
    to_dev_params(vprm, vd);
    std::vector<VioArgs> va(B);
    std::vector<VioSolveArgs> vs(B);
    for (int i = 0; i < B; ++i) {
        VioArgs a{};
        a.img = h->img.p;
        a.cam = h->cam;
        a.pos = h->patch_pos.p;
        a.patch = h->patch_ref.p;
        a.search_level = h->patch_level.p;
        a.Pn = h->Pn;
        a.state = b.states.p + (size_t)i * 5;
        a.prm = vd;
        a.ctrl = b.vio_ctrl.p + i;
        a.force_level = -1;
        a.errors = b.errors.p + (size_t)i * 2 * estride;
        a.err_stride = estride;
        a.partials = b.partials.p + (size_t)i * b.partials_per;
        va[i] = a;
        VioSolveArgs s{};
        s.state = b.states.p + (size_t)i * 5;
        s.state_prop = s.state + 1;
        s.old_state = s.state + 2;
        s.ctrl = b.vio_ctrl.p + i;
        s.prior = b.prior.p + i;
        s.G_last = b.G_last.p + (size_t)i * 108;
        s.partials = a.partials;
        s.nblocks = nb_vio;
        s.errors = a.errors;
        s.err_stride = estride;
        s.Pn_total = h->Pn;
        s.prm = vd;
        s.timeout_flag = &h->barrier.p->timeout;
        vs[i] = s;
    }
    FLB_CUDA(h, cudaMemcpyAsync(b.vio_args.p, va.data(), B * sizeof(VioArgs), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(b.vio_solve.p, vs.data(), B * sizeof(VioSolveArgs), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    {
        LaunchScope lsx(h, FAM_SOLVE);
        k_vio_begin_batched<<<(B + 127) / 128, 128, 0, h->stream>>>(b.vio_ctrl_ptrs.p, B, h->Pn);
        FLB_CUDA(h, cudaGetLastError());
    }
    const int total = 3 * vprm->max_iteration;
    for (int it = 0; it < total; ++it) {
        {
            LaunchScope lsx(h, FAM_VIO);
            k_vio_pass_batched<kVioBlock><<<dim3(nb_vio, B), kVioBlock, 0, h->stream>>>(b.vio_args.p);
            FLB_CUDA(h, cudaGetLastError());
        }
        LaunchScope lsx(h, FAM_SOLVE);
        k_vio_finalize_batched<<<B, kLeaderBlock, 0, h->stream>>>(b.vio_solve.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    return vio_inputs_release(h);
}

int flb_batch_state_download(flb_handle* h, int frame, flb_state18* x, flb_lio_report* lio, flb_vio_report* vio) {
    FLB_CHECK_H(h);
    auto& b = h->batch;
    if (frame < 0 || frame >= b.B) return fail(h, FLB_ERR_INVALID, "flb_batch_state_download: bad frame");
    State18 xs;
    LioCtrl lc;
    VioCtrl vc;
    FLB_CUDA(h, cudaMemcpyAsync(&xs, b.states.p + (size_t)frame * 5, sizeof(State18), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(&lc, b.lio_ctrl.p + frame, sizeof(LioCtrl), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaMemcpyAsync(&vc, b.vio_ctrl.p + frame, sizeof(VioCtrl), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    if (x) std::memcpy(x, &xs, sizeof(State18));
    if (lio) fill_lio_report(lc, lio);
    if (vio) fill_vio_report(vc, vio);
    return FLB_OK;
}

}  // extern "C"

// =======================================================================================
// Device-resident visual map (SURVEY.md section 8 rows f2 / f4)
// =======================================================================================
namespace {

int vm_check(flb_handle* h, const char* who) {
    if (!h->vm.on) return fail(h, FLB_ERR_STATE, "%s: flb_vmap_reset first", who);
    if (!h->cam_set || h->img_w <= 0) return fail(h, FLB_ERR_STATE, "%s: camera and image must be set first", who);
    if (h->cam.width != h->img_w || h->cam.height != h->img_h) return fail(h, FLB_ERR_STATE, "camera / image size mismatch");
    return FLB_OK;
}

// Upload (or derive from the device state) T_f_w of the current frame into vm.pose.
int vm_set_pose(flb_handle* h, const double* Rcw, const double* Pcw) {
    if (Rcw && Pcw) {
        void* stv = nullptr;
        FLB_CUDA(h, h->st_misc.acquire(12 * sizeof(double), &stv));
        double* st = static_cast<double*>(stv);
        std::memcpy(st, Rcw, 9 * sizeof(double));
        std::memcpy(st + 9, Pcw, 3 * sizeof(double));
        FLB_CUDA(h, cudaMemcpyAsync(h->vm.pose.p, st, 12 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        FLB_CUDA(h, h->st_misc.mark(h->stream));
    } else {
        if (!h->state_valid) return fail(h, FLB_ERR_STATE, "visual map: no pose given and no device state");
        { int rcf = flush_state_ops(h); if (rcf) return rcf; }
        LaunchScope ls(h, FAM_OTHER);
        k_vm_pose_from_state<<<1, 32, 0, h->stream>>>(&h->states.p[0], h->vm.rci.p, h->vm.pose.p);
        FLB_CUDA(h, cudaGetLastError());
    }
    return FLB_OK;
}

// points of this call -> vm.pg (packed xyz)
int vm_upload_points(flb_handle* h, const float* xyz, int n, int stride) {
    const size_t n1 = (size_t)std::max(n, 1);
    FLB_CUDA(h, h->vm.pg.reserve(n1 * 3));
    if (n == 0) return FLB_OK;
    void* stv = nullptr;
    FLB_CUDA(h, h->vm.st_pg.acquire(n1 * 3 * sizeof(float), &stv));
    float* st = static_cast<float*>(stv);
    for (int i = 0; i < n; ++i)
        for (int k = 0; k < 3; ++k) {
            const float v = xyz[(size_t)i * stride + k];
            if (!std::isfinite(v) || std::fabs(v) > 5.0e5f) return fail(h, FLB_ERR_INVALID, "visual map: coordinate %d non-finite or beyond 2^20 voxels", i);
            st[3 * (size_t)i + k] = v;
        }
    FLB_CUDA(h, cudaMemcpyAsync(h->vm.pg.p, st, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, h->vm.st_pg.mark(h->stream));
    return FLB_OK;
}

template <typename T>
int vm_grow_buf(flb_handle* h, DevBuf<T>& b, size_t used_ub, size_t need) {
    if (need <= b.cap) return FLB_OK;
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    DevBuf<T> nb;
    FLB_CUDA(h, nb.reserve(std::max(need, b.cap * 2)));
    if (b.p && used_ub) FLB_CUDA(h, cudaMemcpy(nb.p, b.p, std::min(used_ub, b.cap) * sizeof(T), cudaMemcpyDeviceToDevice));
    b.release();
    b = nb;
    return FLB_OK;
}

// Make room for `add_p` more points, `add_f` more features and one more keyframe image.  The host only keeps upper
// bounds of the device counters; when a bound hits the capacity it is refreshed from the device before anything grows.
int vm_ensure_capacity(flb_handle* h, int add_p, int add_f) {
    auto& vm = h->vm;
    const size_t img_bytes = (size_t)h->img_w * h->img_h;
    if ((size_t)(vm.pts_ub + add_p) > vm.pts.cap || (size_t)(vm.fts_ub + add_f) > vm.fts.cap || vm.img_ub + 1 > vm.pool_slots) {
        int c[VM_COUNTERS];
        FLB_CUDA(h, cudaMemcpyAsync(c, vm.counters.p, sizeof(c), cudaMemcpyDeviceToHost, h->stream));
        FLB_CUDA(h, cudaStreamSynchronize(h->stream));
        vm.pts_ub = c[VM_N_POINTS];
        vm.fts_ub = c[VM_N_FEATS];
        vm.img_ub = c[VM_N_IMAGES];
    }
    { int rc = vm_grow_buf(h, vm.pts, (size_t)vm.pts_ub, (size_t)(vm.pts_ub + add_p)); if (rc) return rc; }
    { int rc = vm_grow_buf(h, vm.fts, (size_t)vm.fts_ub, (size_t)(vm.fts_ub + add_f)); if (rc) return rc; }
    if (vm.img_ub + 1 > vm.pool_slots) {
        const int slots = std::max(vm.pool_slots * 2, 16);
        FLB_CUDA(h, cudaStreamSynchronize(h->stream));
        DevBuf<unsigned char> nb;
        FLB_CUDA(h, nb.reserve((size_t)slots * img_bytes));
        if (vm.pool.p && vm.img_ub) FLB_CUDA(h, cudaMemcpy(nb.p, vm.pool.p, (size_t)vm.img_ub * img_bytes, cudaMemcpyDeviceToDevice));
        vm.pool.release();
        vm.pool = nb;
        vm.pool_slots = slots;
    }
    return FLB_OK;
}

}  // namespace

extern "C" {

int flb_vmap_reset(flb_handle* h, const flb_vmap_params* p) {
    FLB_CHECK_H(h);
    if (!p || p->grid_size < 1) return fail(h, FLB_ERR_INVALID, "flb_vmap_reset: bad parameters");
    if (!h->cam_set) return fail(h, FLB_ERR_STATE, "flb_vmap_reset: flb_camera_set first");
    auto& vm = h->vm;
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    VmParams q{};
    q.grid_size = p->grid_size;
    q.grid_n_width = h->cam.width / p->grid_size;                  // :55-57
    q.grid_n_height = h->cam.height / p->grid_size;
    q.length = q.grid_n_width * q.grid_n_height;
    q.halfpatch = 4;
    q.ncc_en = p->ncc_en;
    q.outlier_threshold = p->outlier_threshold;
    q.ncc_thre = p->ncc_thre;
    if (q.length < 1) return fail(h, FLB_ERR_INVALID, "flb_vmap_reset: grid_size larger than the image");
    vm.prm = q;
    {   // Rci / Pci (LidarSelector::init :44-45, set_extrinsic :35-39)
        double Rli[9], Pli[3], t[3];
        m3_T(p->R_LI, Rli);
        m3_vec(Rli, p->t_LI, t);
        for (int i = 0; i < 3; ++i) Pli[i] = -t[i];
        m3_mul(p->Rcl, Rli, vm.Rci_Pci);
        m3_vec(p->Rcl, Pli, t);
        for (int i = 0; i < 3; ++i) vm.Rci_Pci[9 + i] = t[i] + p->Pcl[i];
    }
    const size_t L = (size_t)q.length, npix = (size_t)h->cam.width * h->cam.height;
    FLB_CUDA(h, vm.counters.reserve(VM_COUNTERS));
    FLB_CUDA(h, vm.pose.reserve(12));
    FLB_CUDA(h, vm.rci.reserve(12));
    FLB_CUDA(h, vm.depth.reserve(npix));
    FLB_CUDA(h, vm.cell_best.reserve(L));
    FLB_CUDA(h, vm.cand_key.reserve(L));
    FLB_CUDA(h, vm.cell_type.reserve(L));
    FLB_CUDA(h, vm.map_value.reserve(L));
    FLB_CUDA(h, vm.cell_err.reserve(L));
    FLB_CUDA(h, vm.cell_patch.reserve(L * 192));
    FLB_CUDA(h, vm.sel_error.reserve(L));
    FLB_CUDA(h, vm.cell_flag.reserve(L));
    FLB_CUDA(h, vm.cell_rank.reserve(L));
    FLB_CUDA(h, vm.cell_level.reserve(L));
    FLB_CUDA(h, vm.cell_point.reserve(L));
    FLB_CUDA(h, vm.sel_index.reserve(L));
    FLB_CUDA(h, vm.sel_point.reserve(L));
    FLB_CUDA(h, vm.winner.reserve(L));
    FLB_CUDA(h, vm.scan_tmp.reserve(2 * L));
    FLB_CUDA(h, vm.pts.reserve(std::max<size_t>(4 * L, 1024)));
    FLB_CUDA(h, vm.fts.reserve(std::max<size_t>(8 * L, 2048)));
    // the VIO kernel's inputs are the selection's outputs: one patch per grid cell at most
    FLB_CUDA(h, h->patch_pos.reserve(L * 3));
    FLB_CUDA(h, h->patch_ref.reserve(L * 192));
    FLB_CUDA(h, h->patch_level.reserve(L));
    int c[VM_COUNTERS] = {0};
    c[VM_IMG_FRAME] = -1;
    c[VM_IMG_SLOT] = -1;
    FLB_CUDA(h, cudaMemcpy(vm.counters.p, c, sizeof(c), cudaMemcpyHostToDevice));
    FLB_CUDA(h, cudaMemcpy(vm.rci.p, vm.Rci_Pci, sizeof(vm.Rci_Pci), cudaMemcpyHostToDevice));
    FLB_CUDA(h, cudaMemset(vm.map_value.p, 0, L * sizeof(float)));   // init(), :66
    vm.pts_ub = vm.fts_ub = vm.img_ub = 0;
    vm.on = true;
    return FLB_OK;
}

int flb_vmap_select(flb_handle* h, const double Rcw[9], const double Pcw[3], const float* pg_down, int n, int stride, int* n_selected) {
    FLB_CHECK_H(h);
    { int rc = vm_check(h, "flb_vmap_select"); if (rc) return rc; }
    if (n < 0 || (n > 0 && !pg_down) || stride < 3) return fail(h, FLB_ERR_INVALID, "flb_vmap_select: bad arguments");
    auto& vm = h->vm;
    const int L = vm.prm.length, border = (vm.prm.halfpatch + 1) * 8;
    { int rc = vm_set_pose(h, Rcw, Pcw); if (rc) return rc; }
    { int rc = vm_upload_points(h, pg_down, n, stride); if (rc) return rc; }
    { int rcq = vio_inputs_acquire(h); if (rcq) return rcq; }                 // the current image has landed
    size_t nkeys = 1024;
    while (nkeys < 2 * (size_t)std::max(n, 1)) nkeys <<= 1;
    FLB_CUDA(h, vm.keyset.reserve(nkeys));
    vm.key_mask = (unsigned)(nkeys - 1);
    const size_t npix = (size_t)h->cam.width * h->cam.height;
    // per-patch error buffers of the VIO update that follows: capacity = one patch per grid cell
    FLB_CUDA(h, h->errors.reserve(2 * (size_t)L));
    h->err_stride = std::max(h->err_stride, L);
    FLB_CUDA(h, h->errors.reserve(2 * (size_t)h->err_stride));
    FLB_CUDA(h, h->partials.reserve(std::max<size_t>((size_t)(L / 8 + 2) * kVioPacked, h->partials.cap)));
    {
        LaunchScope ls(h, FAM_OTHER);
        k_vm_clear<<<h->num_sms * 2, 256, 0, h->stream>>>(vm.depth.p, npix, vm.keyset.p, nkeys, vm.cell_best.p, vm.cell_type.p, vm.map_value.p,
                                                          vm.cell_flag.p, L, vm.counters.p);
        if (n > 0)
            k_vm_scan<<<(n + 255) / 256, 256, 0, h->stream>>>(h->cam, vm.pose.p, vm.pg.p, n, border, vm.keyset.p, vm.key_mask, vm.depth.p,
                                                              vm.counters.p);
        const int np = std::max(vm.pts_ub, 1);
        k_vm_candidates<<<(np + 255) / 256, 256, 0, h->stream>>>(h->cam, vm.prm, vm.pose.p, vm.pts.p, vm.counters.p, vm.keyset.p, vm.key_mask,
                                                                 border, vm.cell_best.p, vm.cell_type.p,
                                                                 reinterpret_cast<int*>(vm.map_value.p));
        k_vm_build<<<(L + kVmBuildWarps - 1) / kVmBuildWarps, kVmBuildWarps * 32, 0, h->stream>>>(
            h->cam, vm.prm, vm.pose.p, vm.pts.p, vm.fts.p, vm.pool.p, h->img.p, vm.depth.p, vm.cell_best.p, vm.cell_type.p, vm.counters.p,
            vm.cell_flag.p, vm.cell_level.p, vm.cell_point.p, vm.cell_err.p, vm.cell_patch.p);
        k_vm_rank<<<1, 1024, 0, h->stream>>>(vm.cell_flag.p, L, vm.cell_rank.p, vm.counters.p);
        k_vm_scatter<<<(L + 7) / 8, 256, 0, h->stream>>>(L, vm.cell_flag.p, vm.cell_rank.p, vm.cell_level.p, vm.cell_point.p, vm.cell_err.p,
                                                         vm.cell_patch.p, vm.pts.p, h->patch_pos.p, h->patch_ref.p, h->patch_level.p,
                                                         vm.sel_index.p, vm.sel_point.p, vm.sel_error.p);
        FLB_CUDA(h, cudaGetLastError());
        h->launches += 5;
    }
    { int rcq = vio_inputs_release(h); if (rcq) return rcq; }
    h->pn_on_device = true;
    h->Pn = L;
    h->last_vio_valid = false;
    if (n_selected) {
        int rc = resolve_pn(h);
        if (rc) return rc;
        *n_selected = h->Pn;
    }
    return FLB_OK;
}

int flb_vmap_selected(flb_handle* h, int capacity, int* n_out, int* index, int* point, int* search_level, float* error, double* pos,
                      float* patch) {
    FLB_CHECK_H(h);
    { int rc = vm_check(h, "flb_vmap_selected"); if (rc) return rc; }
    auto& vm = h->vm;
    int n = 0;
    FLB_CUDA(h, cudaMemcpyAsync(&n, vm.counters.p + VM_N_SEL, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    if (n_out) *n_out = n;
    const size_t m = (size_t)std::min(std::max(capacity, 0), n);
    if (m == 0) return FLB_OK;
    cudaStream_t s = h->stream;
    if (index) FLB_CUDA(h, cudaMemcpyAsync(index, vm.sel_index.p, m * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (point) FLB_CUDA(h, cudaMemcpyAsync(point, vm.sel_point.p, m * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (search_level) FLB_CUDA(h, cudaMemcpyAsync(search_level, h->patch_level.p, m * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (error) FLB_CUDA(h, cudaMemcpyAsync(error, vm.sel_error.p, m * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (pos) FLB_CUDA(h, cudaMemcpyAsync(pos, h->patch_pos.p, m * 3 * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (patch) FLB_CUDA(h, cudaMemcpyAsync(patch, h->patch_ref.p, m * 192 * sizeof(float), cudaMemcpyDeviceToHost, s));
    FLB_CUDA(h, cudaStreamSynchronize(s));
    return FLB_OK;
}

int flb_vmap_grow(flb_handle* h, const double Rcw[9], const double Pcw[3], const float* pg, int n, int stride, int frame_id) {
    FLB_CHECK_H(h);
    { int rc = vm_check(h, "flb_vmap_grow"); if (rc) return rc; }
    if (n < 0 || (n > 0 && !pg) || stride < 3 || frame_id < 0) return fail(h, FLB_ERR_INVALID, "flb_vmap_grow: bad arguments");
    auto& vm = h->vm;
    const int L = vm.prm.length, border = (vm.prm.halfpatch + 1) * 8;
    { int rc = vm_ensure_capacity(h, L, L); if (rc) return rc; }
    { int rc = vm_set_pose(h, Rcw, Pcw); if (rc) return rc; }
    { int rc = vm_upload_points(h, pg, n, stride); if (rc) return rc; }
    { int rcq = vio_inputs_acquire(h); if (rcq) return rcq; }
    const size_t img_bytes = (size_t)h->img_w * h->img_h;
    {
        LaunchScope ls(h, FAM_OTHER);
        k_vm_store_image<<<h->num_sms, 256, 0, h->stream>>>(h->img.p, img_bytes, vm.pool.p, vm.counters.p, frame_id);
        k_vmap_seed<<<(L + 255) / 256, 256, 0, h->stream>>>(vm.map_value.p, L, vm.cand_key.p);
        if (n > 0)
            k_vmap_candidates<<<(n + 127) / 128, 128, 0, h->stream>>>(h->cam, vm.pose.p, h->img.p, vm.pg.p, n, vm.prm.grid_size, vm.prm.grid_n_height,
                                                                      border, vm.cand_key.p);
        k_vmap_resolve<<<(L + 255) / 256, 256, 0, h->stream>>>(vm.cand_key.p, L, vm.map_value.p, vm.winner.p);
        k_vm_materialise<<<1, 1024, 0, h->stream>>>(h->cam, L, vm.pose.p, vm.pg.p, vm.winner.p, vm.map_value.p, vm.scan_tmp.p, vm.pts.p, vm.fts.p,
                                                    vm.counters.p, frame_id, (int)vm.pts.cap, (int)vm.fts.cap);
        FLB_CUDA(h, cudaGetLastError());
        h->launches += 4;
    }
    vm.pts_ub += L;
    vm.fts_ub += L;
    vm.img_ub += 1;
    return vio_inputs_release(h);
}

int flb_vmap_add_observations(flb_handle* h, const double Rcw[9], const double Pcw[3], int frame_id) {
    FLB_CHECK_H(h);
    { int rc = vm_check(h, "flb_vmap_add_observations"); if (rc) return rc; }
    if (frame_id < 0) return fail(h, FLB_ERR_INVALID, "flb_vmap_add_observations: bad arguments");
    auto& vm = h->vm;
    const int L = vm.prm.length;
    { int rc = vm_ensure_capacity(h, 0, L); if (rc) return rc; }
    { int rc = vm_set_pose(h, Rcw, Pcw); if (rc) return rc; }
    { int rcq = vio_inputs_acquire(h); if (rcq) return rcq; }
    const size_t img_bytes = (size_t)h->img_w * h->img_h;
    {
        LaunchScope ls(h, FAM_OTHER);
        k_vm_store_image<<<h->num_sms, 256, 0, h->stream>>>(h->img.p, img_bytes, vm.pool.p, vm.counters.p, frame_id);
        k_vm_observe<<<1, 1024, 0, h->stream>>>(h->cam, vm.pose.p, h->img.p, vm.sel_point.p, h->patch_level.p, vm.scan_tmp.p, L, vm.pts.p,
                                                vm.fts.p, vm.counters.p, frame_id, (int)vm.fts.cap);
        FLB_CUDA(h, cudaGetLastError());
        h->launches += 1;
    }
    vm.fts_ub += L;
    vm.img_ub += 1;
    return vio_inputs_release(h);
}

int flb_colorize(flb_handle* h, const double Rcw[9], const double Pcw[3], const uint8_t* bgr, int stride_bytes, const float* world_xyz, int n,
                 int stride, uint8_t* rgb, uint8_t* valid) {
    FLB_CHECK_H(h);
    if (!h->cam_set) return fail(h, FLB_ERR_STATE, "flb_colorize: flb_camera_set first");
    const int W = h->cam.width, H = h->cam.height;
    if (!bgr || stride_bytes < 3 * W || n < 0 || (n > 0 && (!world_xyz || !rgb || !valid)) || stride < 3)
        return fail(h, FLB_ERR_INVALID, "flb_colorize: bad arguments");
    if (n == 0) return FLB_OK;
    auto& vm = h->vm;
    FLB_CUDA(h, vm.pose.reserve(12));
    FLB_CUDA(h, vm.rci.reserve(12));
    if (!(Rcw && Pcw) && !vm.on) return fail(h, FLB_ERR_STATE, "flb_colorize: no pose given and no flb_vmap_reset (extrinsics)");
    { int rc = vm_set_pose(h, Rcw, Pcw); if (rc) return rc; }
    { int rc = vm_upload_points(h, world_xyz, n, stride); if (rc) return rc; }
    const size_t img_bytes = (size_t)W * H * 3;
    FLB_CUDA(h, h->x_rowmask.reserve(img_bytes + (size_t)n * 4));     // colour image | rgb | valid
    unsigned char* d_img = h->x_rowmask.p;
    unsigned char* d_rgb = d_img + img_bytes;
    unsigned char* d_val = d_rgb + (size_t)n * 3;
    void* stv = nullptr;
    FLB_CUDA(h, h->st_img.acquire(img_bytes, &stv));
    unsigned char* st = static_cast<unsigned char*>(stv);
    for (int r = 0; r < H; ++r) std::memcpy(st + (size_t)r * W * 3, bgr + (size_t)r * stride_bytes, (size_t)W * 3);
    FLB_CUDA(h, cudaMemcpyAsync(d_img, st, img_bytes, cudaMemcpyHostToDevice, h->stream));
    FLB_CUDA(h, h->st_img.mark(h->stream));
    {
        LaunchScope ls(h, FAM_OTHER);
        k_vm_colorize<<<(n + 255) / 256, 256, 0, h->stream>>>(h->cam, vm.pose.p, d_img, vm.pg.p, n, d_rgb, d_val);
        FLB_CUDA(h, cudaGetLastError());
    }
    FLB_CUDA(h, h->pin_out.reserve((size_t)n * 4));
    FLB_CUDA(h, cudaMemcpyAsync(h->pin_out.p, d_rgb, (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    std::memcpy(rgb, h->pin_out.p, (size_t)n * 3);
    std::memcpy(valid, static_cast<unsigned char*>(h->pin_out.p) + (size_t)n * 3, n);
    h->last_pass_valid = false;                       // the row-mask export buffer was reused
    return FLB_OK;
}

int flb_vmap_counts(flb_handle* h, int* points, int* features, int* images, int* selected, int* last_added) {
    FLB_CHECK_H(h);
    if (!h->vm.on) return fail(h, FLB_ERR_STATE, "flb_vmap_counts: flb_vmap_reset first");
    int c[VM_COUNTERS];
    FLB_CUDA(h, cudaMemcpyAsync(c, h->vm.counters.p, sizeof(c), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    h->vm.pts_ub = c[VM_N_POINTS];
    h->vm.fts_ub = c[VM_N_FEATS];
    h->vm.img_ub = c[VM_N_IMAGES];
    if (points) *points = c[VM_N_POINTS];
    if (features) *features = c[VM_N_FEATS];
    if (images) *images = c[VM_N_IMAGES];
    if (selected) *selected = c[VM_N_SEL];
    if (last_added) *last_added = c[VM_LAST_ADDED];
    if (c[VM_LAST_ADDED] < 0) return fail(h, FLB_ERR_STATE, "visual map: an append did not fit its buffers (internal capacity bound violated)");
    return FLB_OK;
}

int flb_vmap_map_value(flb_handle* h, float* out, int capacity) {
    FLB_CHECK_H(h);
    if (!h->vm.on || !out) return fail(h, FLB_ERR_STATE, "flb_vmap_map_value: flb_vmap_reset first");
    const size_t n = (size_t)std::min(capacity, h->vm.prm.length);
    FLB_CUDA(h, cudaMemcpyAsync(out, h->vm.map_value.p, n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    FLB_CUDA(h, cudaStreamSynchronize(h->stream));
    return FLB_OK;
}

int flb_vmap_dump(flb_handle* h, int cap_points, int cap_features, double* pos, float* value, int* n_obs, int* obs20, double* ft_geo17,
                  float* ft_score, int* ft_level_id_img) {
    FLB_CHECK_H(h);
    if (!h->vm.on) return fail(h, FLB_ERR_STATE, "flb_vmap_dump: flb_vmap_reset first");
    int np = 0, nf = 0;
    { int rc = flb_vmap_counts(h, &np, &nf, nullptr, nullptr, nullptr); if (rc) return rc; }
    np = std::min(np, cap_points);
    nf = std::min(nf, cap_features);
    std::vector<VmPoint> P((size_t)np);
    std::vector<VmFeature> F((size_t)nf);
    if (np) FLB_CUDA(h, cudaMemcpy(P.data(), h->vm.pts.p, (size_t)np * sizeof(VmPoint), cudaMemcpyDeviceToHost));
    if (nf) FLB_CUDA(h, cudaMemcpy(F.data(), h->vm.fts.p, (size_t)nf * sizeof(VmFeature), cudaMemcpyDeviceToHost));
    for (int j = 0; j < np; ++j) {
        if (pos) std::memcpy(pos + 3 * (size_t)j, P[j].pos, 3 * sizeof(double));
        if (value) value[j] = P[j].value;
        if (n_obs) n_obs[j] = P[j].n_obs;
        if (obs20) for (int q = 0; q < 20; ++q) obs20[20 * (size_t)j + q] = q < P[j].n_obs ? P[j].obs[q] : -1;
    }
    for (int j = 0; j < nf; ++j) {
        if (ft_geo17) {
            double* g = ft_geo17 + 17 * (size_t)j;
            g[0] = F[j].px[0]; g[1] = F[j].px[1];
            std::memcpy(g + 2, F[j].f, 3 * sizeof(double));
            std::memcpy(g + 5, F[j].R, 9 * sizeof(double));
            std::memcpy(g + 14, F[j].t, 3 * sizeof(double));
        }
        if (ft_score) ft_score[j] = F[j].score;
        if (ft_level_id_img) { ft_level_id_img[3 * (size_t)j] = F[j].level; ft_level_id_img[3 * (size_t)j + 1] = F[j].id; ft_level_id_img[3 * (size_t)j + 2] = F[j].img; }
    }
    return FLB_OK;
}

}  // extern "C"
