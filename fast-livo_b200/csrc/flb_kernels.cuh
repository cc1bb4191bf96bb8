// flb_kernels.cuh -- __global__ kernels of the FAST-LIVO hot path for sm_100a.
//
// Kernel families (SURVEY.md §8):
//   * LIO pass  : per-point world transform + exact 5-NN over the device map grid + float32 QR
//                 plane fit (rematch passes) + point-to-plane residual + Jacobian row + H^T H / H^T z
//   * VIO pass  : warp-per-patch photometric residual + d r / d xi over 8x8 pixels + H^T H / H^T z
//   * leader    : fixed-order cross-block reduction, the 18-DoF iterated-ESKF step, state [+],
//                 convergence / rematch / stop control -- all on the device
//   * map / scan preparation (cell sort, Morton sort)
// Two execution modes share all of the above:
//   persistent      one cooperative launch per update: worker blocks run the passes, ONE leader block (no
//                   points / patches of its own) reduces, solves and publishes the next pose as a flagged
//                   packet the workers poll (k_lio_update_persistent / k_vio_update_persistent)
//   kernel-per-pass k_*_pass + k_*_finalize (one block running the same leader code); with blockIdx.y = frame the same
//                   bodies are the batched-frames kernels (k_*_pass_batched / k_*_finalize_batched)
// What sits OFF the critical path of a VIO pass (DESIGN.md section 4.3): the exact sequential float sum over the
// per-patch errors (the leader publishes the accept branch before it is known and discards the running pass if it
// says "reject") and the exact 64-step chain inside a patch (run by the worker after its block has arrived; the leader
// polls self-validating {tag : error} units).  Multi-GPU: the same units and 16-byte {payload, tag} lines written
// straight into the peers' mailboxes over NVLink (p2p_exchange), no separate flag, no fence.
// No tensor cores: nothing here is a dense contraction.  No floating-point atomics: every reduction
// has a fixed order, so results are bit-reproducible run to run and identical across ranks.
#pragma once

#include <cuda_runtime.h>
#include <cub/block/block_radix_sort.cuh>
#include "flb_device.cuh"

namespace flb {

// After an L2 flush (or simply other work) the first pass of a frame finds neither its data nor the translations of
// its pages cached, and it discovers the pages one dependent step at a time (scan -> cell table -> map points ->
// plane cache ...).  The leader block, idle until the first pass arrives, touches one word of every 2 MB page of every
// buffer the update will use, all at once, so the page walks overlap instead of queueing behind each other.
struct WarmList {
    const void* p[10];
    unsigned long long bytes[10];
    int n;
};
__device__ __forceinline__ void warm_pages(const WarmList& w, int tid, int nt) {
    constexpr unsigned long long kPage = 2ull << 20;
    int slot = 0;
    for (int b = 0; b < w.n; ++b) {
        const char* base = static_cast<const char*>(w.p[b]);
        if (!base) continue;
        const unsigned long long npages = (w.bytes[b] + kPage - 1) / kPage;
        for (unsigned long long pg = 0; pg < npages; ++pg, ++slot)
            if (slot % nt == tid) {
                const unsigned long long off = pg * kPage;
                unsigned v;
                asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(v) : "l"(base + (off < w.bytes[b] ? (off & ~3ull) : 0ull)) : "memory");
            }
    }
}

// ---------------------------------------------------------------------------------------
// device-resident control blocks
// ---------------------------------------------------------------------------------------
struct LioCtrl {
    // loop state, src/laserMapping.cpp:1472-1473, 1506, 1634-1635, 1700-1731
    int iterCount;
    int rematch_num;
    int nearest_search_en;
    int stop;
    // report
    int passes, knn_passes, n_eff_last, converged_last, status;
    double res_mean_last;
    long long rows_total;
};

struct VioCtrl {
    int level;          // 2,1,0 ; -1 when finished
    int iteration;
    int stop;
    float last_error;   // per level
    float now_error;
    int any_solved;     // G valid
    int passes[3];
    float level_error[3];
    long long rows_total;
    int skipped_last, cov_updated, status;
    int err_buf;        // which half of the double-buffered per-patch errors the last executed pass wrote
};

struct LioParamsDev {
    double R_LI[9], t_LI[3];
    double sigma;
    int max_iteration;
    double conv_rot_deg, conv_pos_cm;
};

struct VioParamsDev {
    double Rci[9], Pci[3];
    double Jdphi_dR[9], Jdp_dR[9];   // state-independent Jacobian factors (LidarSelector::init)
    double sigma;
    int max_iteration;
    float conv_rot_deg, conv_pos_cm;
    int force_all_passes;
    int single_level;                // UpdateState alone (one pyramid level, :743-902): stop when the level ends, no :980
};

// Packed sizes: W(W+1)/2 upper-triangular products + W (H^T z) + 2 scalars.
__host__ __device__ constexpr int lio_packed(int W) { return W * (W + 1) / 2 + W + 2; }
constexpr int kVioPacked = 21 + 6 + 2;  // + n_meas, skipped

constexpr int kLioBlock = 128;          // kernel-per-pass / IKFoM kernels
constexpr int kVioBlock = 256;
constexpr int kLioPersBlock = 256;      // persistent kernels: one block per SM (half the partials and
constexpr int kVioPersBlock = 512;      // arrive tickets of two smaller blocks; same warps per SM)
constexpr int kLeaderBlock = 256;       // block size of the kernel-per-pass finalize kernels

// Optional device-side pass trace (profiling aid): %globaltimer (ns) at kernel entry [0], then for
// pass k: [1+2k] = all blocks arrived (leader elected), [2+2k] = leader released the barrier.
constexpr int kTraceLen = 128;
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

// Transposing butterfly reduction of up to 32 per-lane accumulators: after 5 exchange steps lane l holds
// the warp-wide total of accumulator l.  31 double shuffles instead of 5 per accumulator (K = 29: 145);
// fixed tree => deterministic.
template <int N, int S>
struct ButterflyStep {
    static __device__ __forceinline__ void run(double (&v)[32], int lane) {
        constexpr int H = N / 2;
        const bool up = (lane & S) != 0;
#pragma unroll
        for (int j = 0; j < H; ++j) {
            const double keep = up ? v[j + H] : v[j];
            const double send = up ? v[j] : v[j + H];
            v[j] = keep + __shfl_xor_sync(0xffffffffu, send, S);
        }
        ButterflyStep<H, S / 2>::run(v, lane);
    }
};
template <int N>
struct ButterflyStep<N, 0> {
    static __device__ __forceinline__ void run(double (&)[32], int) {}
};
template <int K>
__device__ __forceinline__ double warp_transpose_reduce(const double (&acc)[K]) {
    static_assert(K <= 32, "at most 32 accumulators");
    double v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = (i < K) ? acc[i] : 0.0;
    ButterflyStep<32, 16>::run(v, threadIdx.x & 31);
    return v[0];
}

// ---------------------------------------------------------------------------------------
// map grid build
// ---------------------------------------------------------------------------------------
__global__ void k_map_cell_ids(const float* __restrict__ xyz, int M, int stride, GridDesc g, unsigned* __restrict__ keys,
                               int* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const float x = xyz[(size_t)i * stride], y = xyz[(size_t)i * stride + 1], z = xyz[(size_t)i * stride + 2];
    int cx = (int)floorf((x - g.ox) * g.inv_cell), cy = (int)floorf((y - g.oy) * g.inv_cell),
        cz = (int)floorf((z - g.oz) * g.inv_cell);
    cx = min(max(cx, 0), g.nx - 1);
    cy = min(max(cy, 0), g.ny - 1);
    cz = min(max(cz, 0), g.nz - 1);
    keys[i] = (unsigned)((cz * g.ny + cy) * g.nx + cx);
    vals[i] = i;
}

// After the stable sort by cell: gather points (w = original index bits) and mark cell starts.
__global__ void k_map_gather(const float* __restrict__ xyz, int M, int stride, const int* __restrict__ vals_sorted,
                             float4* __restrict__ pts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const int src = vals_sorted[i];
    float4 p;
    p.x = xyz[(size_t)src * stride];
    p.y = xyz[(size_t)src * stride + 1];
    p.z = xyz[(size_t)src * stride + 2];
    p.w = __int_as_float(src);
    pts[i] = p;
}

// cell_start[c] = first sorted position whose cell id is >= c (c = 0 .. ncell): one binary search per cell, so long
// runs of empty cells (a map that covers little of its bounding box) cost nothing extra.
__device__ __forceinline__ int lower_bound_u32(const unsigned* __restrict__ a, int n, unsigned v) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}
__global__ void k_cell_starts(const unsigned* __restrict__ keys_sorted, int M, int* __restrict__ cell_start, int ncell) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > ncell) return;
    cell_start[c] = lower_bound_u32(keys_sorted, M, (unsigned)c);
}

// bounding box of n packed xyz points: ordered-int atomics into box[6] = {min x, y, z, max x, y, z} (as ordered bits)
__device__ __forceinline__ int f32_ordered_int(float f) {
    const int b = __float_as_int(f);
    return b >= 0 ? b : (b ^ 0x7fffffff);
}
__global__ void k_bbox(const float* __restrict__ xyz, int n, int* __restrict__ box) {
    int mn[3] = {0x7fffffff, 0x7fffffff, 0x7fffffff}, mx[3] = {(int)0x80000000, (int)0x80000000, (int)0x80000000};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const int v = f32_ordered_int(xyz[3 * (size_t)i + a]);
            mn[a] = min(mn[a], v);
            mx[a] = max(mx[a], v);
        }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        for (int o = 16; o > 0; o >>= 1) {
            mn[a] = min(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
            mx[a] = max(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(box + a, mn[a]);
            atomicMax(box + 3 + a, mx[a]);
        }
    }
}

// ---------------------------------------------------------------------------------------
// map maintenance (SURVEY.md section 8 row f1): KD_TREE::Add_Points(points, downsample = true)
// (include/ikd-Tree/ikd_Tree.cpp:382-457) and Delete_Point_Boxes (:501-521) on the device map.
//
// Add_Points processes the new points one by one: box = the downsample voxel of the point,
// Downsample_Storage = live points in the box, result = the one closest to the voxel centre (strict <,
// starting from the new point); if the box held more than one point, or the new point won, the box is
// emptied and `result` put back.  Its net effect per voxel is order-independent up to ties, so the
// device version sorts (existing + new) points by voxel and lets one thread replay that sequential
// rule over each voxel's handful of points.
//
// That holds only while every point lies in exactly one float box.  The box of voxel k is
// [fl(k*ds), fl(fl(k*ds) + ds)) per axis, so for a ds that is not a power of two neighbouring boxes can
// overlap or leave a gap of an ulp: a point within a few ulps of a boundary can lie in two boxes, or in
// none (not even its own).  Its fate then depends on the order in which the reference meets the points.
// So a voxel is resolved in parallel only when it is "clean": every point involved lies in its own box
// and in no neighbour's (vox_clean).  The other voxels ("dirty": a point lands within a few ulps of a
// boundary about once in 10^4..10^5 per axis, so a real frame has none or a handful) are replayed by one
// thread in submission order with the reference's sequential rule and its exact box test.
// ---------------------------------------------------------------------------------------
// p lies strictly in its own float box (ikd_Tree.cpp:392-397, half-open test of :998) and in no neighbour's
__device__ __forceinline__ bool vox_clean(const float* p, float ds) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float kf = floorf(p[a] / ds);
#pragma unroll
        for (int d = -1; d <= 1; ++d) {
            const float mn = __fmul_rn(kf + (float)d, ds), mx = __fadd_rn(mn, ds);
            const bool in = mn <= p[a] && mx > p[a];
            if (in != (d == 0)) return false;
        }
    }
    return true;
}
__device__ __forceinline__ bool in_vox_box(const float* mn, const float* mx, float x, float y, float z) {
    return mn[0] <= x && mx[0] > x && mn[1] <= y && mx[1] > y && mn[2] <= z && mx[2] > z;
}
// box and centre of the downsample voxel of p, float arithmetic as ikd_Tree.cpp:392-400 writes it
__device__ __forceinline__ void vox_box(const float* p, float ds, float* mn, float* mx, float* mid) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        mn[a] = __fmul_rn(floorf(p[a] / ds), ds);
        mx[a] = __fadd_rn(mn[a], ds);
        mid[a] = (float)((double)mn[a] + (double)(mx[a] - mn[a]) / 2.0);
    }
}
// the few dirty entries, sorted in place by `by[entry]` (submission order); one thread
__device__ void sort_small_by(int* e, int n, const int* by) {
    for (int i = 1; i < n; ++i) {
        const int v = e[i];
        int j = i - 1;
        while (j >= 0 && (by ? by[e[j]] : e[j]) > (by ? by[v] : v)) { e[j + 1] = e[j]; --j; }
        e[j + 1] = v;
    }
}
__device__ __forceinline__ unsigned long long vox_key(float x, float y, float z, float ds) {
    // floor(p / downsample_size) per axis (ikd_Tree.cpp:392-396), biased into 21 bits each
    const long long ix = (long long)floorf(x / ds) + (1ll << 20), iy = (long long)floorf(y / ds) + (1ll << 20),
                    iz = (long long)floorf(z / ds) + (1ll << 20);
    return ((unsigned long long)(iz & 0x1fffff) << 42) | ((unsigned long long)(iy & 0x1fffff) << 21) |
           (unsigned long long)(ix & 0x1fffff);
}

__global__ void k_vox_keys(const float* __restrict__ xyz, int total, float ds, unsigned long long* __restrict__ keys,
                           int* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    keys[i] = vox_key(xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2], ds);
    vals[i] = i;
}

// sorted positions of the points (existing and new) that are not clean; counts[0] must be zero on entry
__global__ void k_vox_unclean(const int* __restrict__ vals, const float* __restrict__ xyz, int total, float ds,
                              int* __restrict__ unclean, int* __restrict__ counts) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= total) return;
    if (!vox_clean(xyz + 3 * (size_t)vals[j], ds)) unclean[atomicAdd(counts, 1)] = j;
}

// keys/vals sorted by voxel (stable: ascending index inside a voxel, so existing points [idx < M] come
// first and new points keep their submission order).  One thread per voxel segment.  A dirty voxel keeps its
// existing points, drops its new ones for now and queues them in rep[] for k_vox_replay (counts[1]).
__global__ void k_vox_resolve(const unsigned long long* __restrict__ keys, const int* __restrict__ vals,
                              const float* __restrict__ xyz, int total, int M, float ds, const int* __restrict__ unclean,
                              int* __restrict__ counts, int* __restrict__ rep, unsigned char* __restrict__ keep) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const unsigned long long k = keys[i];
    if (i > 0 && keys[i - 1] == k) return;          // not a segment head
    int end = i;
    while (end < total && keys[end] == k) ++end;
    int first_new = end;
    for (int j = i; j < end; ++j)
        if (vals[j] >= M) { first_new = j; break; }
    if (first_new == end) {                         // voxel untouched by this batch: keep everything
        for (int j = i; j < end; ++j) keep[j] = 1;
        return;
    }
    // box and centre from the first new point (ikd_Tree.cpp:392-400), float arithmetic as written there
    const int v0 = vals[first_new];
    float mn[3], mx[3], mid[3];
    vox_box(xyz + 3 * (size_t)v0, ds, mn, mx, mid);
    // dirty: a point of the voxel outside its box or inside a neighbour's, or a point of another voxel inside this box
    bool dirty = false;
    for (int j = i; j < end && !dirty; ++j) dirty = !vox_clean(xyz + 3 * (size_t)vals[j], ds);
    const int nu = counts[0];
    for (int u = 0; u < nu && !dirty; ++u) {
        const float* p = xyz + 3 * (size_t)vals[unclean[u]];
        dirty = in_vox_box(mn, mx, p[0], p[1], p[2]);
    }
    if (dirty) {
        for (int j = i; j < end; ++j) {
            keep[j] = vals[j] < M ? 1 : 0;
            if (vals[j] >= M) rep[atomicAdd(counts + 1, 1)] = j;
        }
        return;
    }
    // content of the box: existing points that pass the half-open box test (:1001)
    int c = 0, best = -1;
    float best_d = INFINITY;
    for (int j = i; j < first_new; ++j) {
        const float* p = xyz + 3 * (size_t)vals[j];
        const bool in = mn[0] <= p[0] && mx[0] > p[0] && mn[1] <= p[1] && mx[1] > p[1] && mn[2] <= p[2] && mx[2] > p[2];
        keep[j] = in ? 0 : 1;                       // (a point just outside its own float box is never touched)
        if (in) {
            ++c;
            const float d = dist2f(p[0], p[1], p[2], mid[0], mid[1], mid[2]);
            if (d < best_d) { best_d = d; best = j; }
        }
    }
    const int c0 = c, best0 = best;
    bool replaced = false;
    for (int j = first_new; j < end; ++j) {
        keep[j] = 0;
        const float* p = xyz + 3 * (size_t)vals[j];
        const float d = dist2f(p[0], p[1], p[2], mid[0], mid[1], mid[2]);
        const bool p_wins = !(best_d < d);          // tmp_dist < min_dist, strict (:405)
        if (c > 1 || p_wins) {                      // :412
            if (p_wins) { best = j; best_d = d; }
            c = 1;
            replaced = true;
        }
    }
    if (replaced) {
        keep[best] = 1;
    } else if (c0 > 0) {
        // the single existing point beat every new one: nothing changes (:412 false every time)
        for (int j = i; j < first_new; ++j)
            if (!keep[j]) keep[j] = 1;
        (void)best0;
    }
}

// The new points of the dirty voxels, one at a time in submission order, with the reference's sequential rule
// (ikd_Tree.cpp:390-418).  The live points of a dirty voxel's box are those of its own key segment that pass the box
// test, plus unclean points of other voxels that do (a clean point lies in its own box only).  One thread.
__global__ void k_vox_replay(const unsigned long long* __restrict__ keys, const int* __restrict__ vals, const float* __restrict__ xyz,
                             int total, float ds, const int* __restrict__ unclean, int* __restrict__ counts, int* __restrict__ rep,
                             unsigned char* __restrict__ keep) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const int nr = counts[1], nu = counts[0];
    if (nr == 0) return;
    sort_small_by(rep, nr, vals);
    for (int r = 0; r < nr; ++r) {
        const int j = rep[r];
        const float* p = xyz + 3 * (size_t)vals[j];
        float mn[3], mx[3], mid[3];
        vox_box(p, ds, mn, mx, mid);
        const unsigned long long k = keys[j];
        int s0 = j, s1 = j + 1;
        while (s0 > 0 && keys[s0 - 1] == k) --s0;
        while (s1 < total && keys[s1] == k) ++s1;
        // two sweeps over Downsample_Storage: count + closest, then (if the box changes) delete all but the result
        int c = 0, best = j;
        float best_d = dist2f(p[0], p[1], p[2], mid[0], mid[1], mid[2]);
        for (int pass = 0; pass < 2; ++pass) {
            const bool del = pass == 1;
            if (del && !(c > 1 || best == j)) break;                       // :412 false: nothing changes
            for (int t = s0; t < s1 + nu; ++t) {
                const int q = t < s1 ? t : unclean[t - s1];
                if (!keep[q] || (t >= s1 && keys[q] == k)) continue;       // dead, or already seen in the segment
                const float* o = xyz + 3 * (size_t)vals[q];
                if (!in_vox_box(mn, mx, o[0], o[1], o[2])) continue;
                if (del) { keep[q] = 0; continue; }
                ++c;
                const float d = dist2f(o[0], o[1], o[2], mid[0], mid[1], mid[2]);
                if (d < best_d) { best_d = d; best = q; }
            }
            if (del) keep[best] = 1;
        }
    }
}

// keep = not inside any box (half-open test of Delete_by_range, ikd_Tree.cpp:650); vals = iota
__global__ void k_box_flags(const float* __restrict__ xyz, int M, const float* __restrict__ boxes, int nb,
                            unsigned char* __restrict__ keep, int* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const float x = xyz[3 * (size_t)i], y = xyz[3 * (size_t)i + 1], z = xyz[3 * (size_t)i + 2];
    bool del = false;
    for (int b = 0; b < nb; ++b) {
        const float* q = boxes + 6 * b;
        if (q[0] <= x && q[3] > x && q[1] <= y && q[4] > y && q[2] <= z && q[5] > z) del = true;
    }
    keep[i] = del ? 0 : 1;
    vals[i] = i;
}

__global__ void k_gather_xyz(const float* __restrict__ src, const int* __restrict__ idx, int n, float* __restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int s = idx[i];
    dst[3 * (size_t)i] = src[3 * (size_t)s];
    dst[3 * (size_t)i + 1] = src[3 * (size_t)s + 1];
    dst[3 * (size_t)i + 2] = src[3 * (size_t)s + 2];
}

// ---------------------------------------------------------------------------------------
// Incremental Add_Points: only the voxels the NEW points fall into are looked at.  The new points are sorted by
// downsample voxel; one thread per touched voxel finds the live points of its box through the kNN grid (a box overlaps
// at most a handful of cells), replays the reference's sequential rule, marks the existing points that go and the one
// new point that stays; the sorted grid is then MERGED (live existing points keep their order, inserts are appended to
// their cells) instead of being re-sorted.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ int grid_axis_cell(float v, float o, float inv_cell, int n) {
    const int c = (int)floorf((v - o) * inv_cell);
    return min(max(c, 0), n - 1);
}
// also lists the new points that are not clean (unclean[], counts[0]: zero on entry)
__global__ void k_vox_keys_rel(const float* __restrict__ xyz, int n, float ds, int bx, int by, int bz, int sy, int sz,
                               unsigned long long* __restrict__ keys, int* __restrict__ vals, int* __restrict__ unclean,
                               int* __restrict__ counts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (!vox_clean(xyz + 3 * (size_t)i, ds)) unclean[atomicAdd(counts, 1)] = i;
    // floor(p / ds) per axis (ikd_Tree.cpp:392-396) relative to the map box, packed x | y << sy | z << sz
    const long long ix = (long long)floorf(xyz[3 * (size_t)i] / ds) - bx, iy = (long long)floorf(xyz[3 * (size_t)i + 1] / ds) - by,
                    iz = (long long)floorf(xyz[3 * (size_t)i + 2] / ds) - bz;
    keys[i] = (unsigned long long)ix | ((unsigned long long)iy << sy) | ((unsigned long long)iz << sz);
    vals[i] = i;
}
__global__ void k_vox_resolve_incremental(const unsigned long long* __restrict__ keys, const int* __restrict__ vals,
                                          const float* __restrict__ nxyz, int n, float ds, GridDesc g, const int* __restrict__ cell_start,
                                          const float4* __restrict__ pts, const int* __restrict__ unclean, int* __restrict__ counts,
                                          int* __restrict__ rep, unsigned char* __restrict__ dead, unsigned char* __restrict__ ins) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long k = keys[i];
    if (i > 0 && keys[i - 1] == k) return;          // not a segment head
    int end = i;
    while (end < n && keys[end] == k) ++end;
    const int v0 = vals[i];
    float mn[3], mx[3], mid[3];
    vox_box(nxyz + 3 * (size_t)v0, ds, mn, mx, mid);
    // dirty (see vox_clean): a new point of the voxel, or any point found in its box, is not clean
    bool dirty = false;
    for (int j = i; j < end && !dirty; ++j) dirty = !vox_clean(nxyz + 3 * (size_t)vals[j], ds);
    const int nu = counts[0];
    for (int u = 0; u < nu && !dirty; ++u) {
        const float* p = nxyz + 3 * (size_t)unclean[u];
        dirty = in_vox_box(mn, mx, p[0], p[1], p[2]);
    }
    // Downsample_Storage = live points in the half-open box (Search_by_range, :1001)
    const int cx0 = grid_axis_cell(mn[0], g.ox, g.inv_cell, g.nx), cx1 = grid_axis_cell(mx[0], g.ox, g.inv_cell, g.nx);
    const int cy0 = grid_axis_cell(mn[1], g.oy, g.inv_cell, g.ny), cy1 = grid_axis_cell(mx[1], g.oy, g.inv_cell, g.ny);
    const int cz0 = grid_axis_cell(mn[2], g.oz, g.inv_cell, g.nz), cz1 = grid_axis_cell(mx[2], g.oz, g.inv_cell, g.nz);
    int c = 0, best = -1;                           // best >= 0: sorted position of an existing point; <= -2: -(j + 2) of a new one
    float best_d = INFINITY;
    for (int z = cz0; z <= cz1; ++z)
        for (int y = cy0; y <= cy1; ++y) {
            const int row = (z * g.ny + y) * g.nx;
            const int s0 = cell_start[row + cx0], s1 = cell_start[row + cx1 + 1];
            for (int m = s0; m < s1; ++m) {
                const float4 p = pts[m];
                if (mn[0] <= p.x && mx[0] > p.x && mn[1] <= p.y && mx[1] > p.y && mn[2] <= p.z && mx[2] > p.z) {
                    ++c;
                    const float d = dist2f(p.x, p.y, p.z, mid[0], mid[1], mid[2]);
                    if (d < best_d) { best_d = d; best = m; }
                    const float o[3] = {p.x, p.y, p.z};
                    dirty = dirty || !vox_clean(o, ds);
                }
            }
        }
    if (dirty) {                                    // leave the voxel to k_vox_replay_incremental
        for (int j = i; j < end; ++j) rep[atomicAdd(counts + 1, 1)] = vals[j];
        return;
    }
    bool replaced = false;
    for (int j = i; j < end; ++j) {
        const float* p = nxyz + 3 * (size_t)vals[j];
        const float d = dist2f(p[0], p[1], p[2], mid[0], mid[1], mid[2]);
        const bool p_wins = !(best_d < d);          // tmp_dist < min_dist, strict (:405)
        if (c > 1 || p_wins) {                      // :412
            if (p_wins) { best = -(j + 2); best_d = d; }
            c = 1;
            replaced = true;
        }
    }
    if (!replaced) return;                          // the single existing point beat every new one: nothing changes
    for (int z = cz0; z <= cz1; ++z)
        for (int y = cy0; y <= cy1; ++y) {
            const int row = (z * g.ny + y) * g.nx;
            const int s0 = cell_start[row + cx0], s1 = cell_start[row + cx1 + 1];
            for (int m = s0; m < s1; ++m) {
                const float4 p = pts[m];
                if (m != best && mn[0] <= p.x && mx[0] > p.x && mn[1] <= p.y && mx[1] > p.y && mn[2] <= p.z && mx[2] > p.z) dead[m] = 1;
            }
        }
    if (best <= -2) ins[vals[-(best + 2)]] = 1;
}
// The new points of the dirty voxels, one at a time in submission order, with the reference's sequential rule
// (ikd_Tree.cpp:390-418): Downsample_Storage = live existing points of the box (through the grid) + new points the
// replay has kept so far that lie in it (no clean voxel's point can: it lies in its own box only).  One thread.
__global__ void k_vox_replay_incremental(const float* __restrict__ nxyz, float ds, GridDesc g, const int* __restrict__ cell_start,
                                         const float4* __restrict__ pts, int* __restrict__ counts, int* __restrict__ rep,
                                         unsigned char* __restrict__ dead, unsigned char* __restrict__ ins) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const int nr = counts[1];
    if (nr == 0) return;
    sort_small_by(rep, nr, nullptr);
    for (int r = 0; r < nr; ++r) {
        const int v = rep[r];
        const float* p = nxyz + 3 * (size_t)v;
        float mn[3], mx[3], mid[3];
        vox_box(p, ds, mn, mx, mid);
        const int cx0 = grid_axis_cell(mn[0], g.ox, g.inv_cell, g.nx), cx1 = grid_axis_cell(mx[0], g.ox, g.inv_cell, g.nx);
        const int cy0 = grid_axis_cell(mn[1], g.oy, g.inv_cell, g.ny), cy1 = grid_axis_cell(mx[1], g.oy, g.inv_cell, g.ny);
        const int cz0 = grid_axis_cell(mn[2], g.oz, g.inv_cell, g.nz), cz1 = grid_axis_cell(mx[2], g.oz, g.inv_cell, g.nz);
        int c = 0, best = -(v + 2);                 // >= 0: sorted position of an existing point; <= -2: -(index + 2) of a new one
        float best_d = dist2f(p[0], p[1], p[2], mid[0], mid[1], mid[2]);
        for (int pass = 0; pass < 2; ++pass) {
            const bool del = pass == 1;
            if (del && !(c > 1 || best == -(v + 2))) break;              // :412 false: nothing changes
            for (int z = cz0; z <= cz1; ++z)
                for (int y = cy0; y <= cy1; ++y) {
                    const int row = (z * g.ny + y) * g.nx;
                    const int s0 = cell_start[row + cx0], s1 = cell_start[row + cx1 + 1];
                    for (int m = s0; m < s1; ++m) {
                        const float4 q = pts[m];
                        if (dead[m] || !in_vox_box(mn, mx, q.x, q.y, q.z)) continue;
                        if (del) { dead[m] = 1; continue; }
                        ++c;
                        const float d = dist2f(q.x, q.y, q.z, mid[0], mid[1], mid[2]);
                        if (d < best_d) { best_d = d; best = m; }
                    }
                }
            for (int t = 0; t < r; ++t) {
                const int u = rep[t];
                const float* q = nxyz + 3 * (size_t)u;
                if (!ins[u] || !in_vox_box(mn, mx, q[0], q[1], q[2])) continue;
                if (del) { ins[u] = 0; continue; }
                ++c;
                const float d = dist2f(q[0], q[1], q[2], mid[0], mid[1], mid[2]);
                if (d < best_d) { best_d = d; best = -(u + 2); }
            }
            if (del) {
                if (best >= 0) dead[best] = 0;
                else ins[-(best + 2)] = 1;
            }
        }
    }
}
// cell id of every new point (ncell = "not inserted": sorts behind every real cell)
__global__ void k_insert_cells(const float* __restrict__ nxyz, int n, const unsigned char* __restrict__ ins, GridDesc g, int ncell,
                               unsigned* __restrict__ keys, int* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned key = (unsigned)ncell;
    if (ins[i]) {
        const int cx = grid_axis_cell(nxyz[3 * (size_t)i], g.ox, g.inv_cell, g.nx), cy = grid_axis_cell(nxyz[3 * (size_t)i + 1], g.oy, g.inv_cell, g.ny),
                  cz = grid_axis_cell(nxyz[3 * (size_t)i + 2], g.oz, g.inv_cell, g.nz);
        key = (unsigned)((cz * g.ny + cy) * g.nx + cx);
    }
    keys[i] = key;
    vals[i] = i;
}
__global__ void k_dead_to_int(const unsigned char* __restrict__ dead, int M, int* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < M) out[i] = dead[i];
}
// counts[0] = dead points, counts[1] = inserted points (needs dead_before of the last element + its flag)
__global__ void k_merge_counts(const int* __restrict__ dead_before, const unsigned char* __restrict__ dead, int M,
                               const unsigned* __restrict__ ins_keys_sorted, int n, int ncell, int* __restrict__ counts) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        counts[0] = dead_before[M - 1] + dead[M - 1];
        counts[1] = lower_bound_u32(ins_keys_sorted, n, (unsigned)ncell);
    }
}
__global__ void k_merge_cell_starts(const int* __restrict__ cs_old, const int* __restrict__ dead_before, const int* __restrict__ counts,
                                    int M, const unsigned* __restrict__ ins_keys_sorted, int n, int ncell, int* __restrict__ cs_new) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > ncell) return;
    const int s = cs_old[c];
    const int db = s < M ? dead_before[s] : counts[0];
    cs_new[c] = s - db + lower_bound_u32(ins_keys_sorted, n, (unsigned)c);
}
__global__ void k_merge_existing(const float4* __restrict__ pts_old, const unsigned char* __restrict__ dead,
                                 const int* __restrict__ dead_before, int M, GridDesc g, const unsigned* __restrict__ ins_keys_sorted, int n,
                                 float4* __restrict__ pts_new, float* __restrict__ raw_new) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M || dead[m]) return;
    float4 p = pts_old[m];
    const int cx = grid_axis_cell(p.x, g.ox, g.inv_cell, g.nx), cy = grid_axis_cell(p.y, g.oy, g.inv_cell, g.ny),
              cz = grid_axis_cell(p.z, g.oz, g.inv_cell, g.nz);
    const unsigned cell = (unsigned)((cz * g.ny + cy) * g.nx + cx);
    const int pos = m - dead_before[m] + lower_bound_u32(ins_keys_sorted, n, cell);
    p.w = __int_as_float(pos);
    pts_new[pos] = p;
    raw_new[3 * (size_t)pos] = p.x; raw_new[3 * (size_t)pos + 1] = p.y; raw_new[3 * (size_t)pos + 2] = p.z;
}
__global__ void k_merge_inserts(const float* __restrict__ nxyz, const unsigned* __restrict__ ins_keys_sorted, const int* __restrict__ ins_vals_sorted,
                                int n, const int* __restrict__ counts, const int* __restrict__ cs_new, float4* __restrict__ pts_new,
                                float* __restrict__ raw_new) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= counts[1]) return;
    const unsigned cell = ins_keys_sorted[k];
    const int first = lower_bound_u32(ins_keys_sorted, n, cell), last = lower_bound_u32(ins_keys_sorted, n, cell + 1u);
    const int pos = cs_new[cell + 1] - (last - first) + (k - first);     // inserts go behind the cell's surviving points
    const float* q = nxyz + 3 * (size_t)ins_vals_sorted[k];
    pts_new[pos] = make_float4(q[0], q[1], q[2], __int_as_float(pos));
    raw_new[3 * (size_t)pos] = q[0]; raw_new[3 * (size_t)pos + 1] = q[1]; raw_new[3 * (size_t)pos + 2] = q[2];
}

// ---------------------------------------------------------------------------------------
// pcl::VoxelGrid<PointType> (centroid per leaf; src/laserMapping.cpp:1398-1399 downSizeFilterSurf, src/lidar_selection.cpp:7,
// :351-352 downSizeFilter): leaf index as PCL forms it (min_b from the cloud's minimum, idx = ijk . divb_mul), points of a
// leaf summed in float in their ORIGINAL ORDER (PCL's own order inside a leaf is that of an unstable std::sort: unspecified),
// output in ascending leaf index like PCL.  box = k_bbox's ordered-int {min, max}.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float ordered_int_f32(int v) { return __int_as_float(v >= 0 ? v : (v ^ 0x7fffffff)); }
__global__ void k_vg_keys(const float* __restrict__ xyz, int n, const int* __restrict__ box, float inv_leaf, unsigned* __restrict__ keys,
                          int* __restrict__ vals, int* __restrict__ status) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int min_b[3], div_b[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        min_b[a] = (int)floorf(ordered_int_f32(box[a]) * inv_leaf);
        div_b[a] = (int)floorf(ordered_int_f32(box[3 + a]) * inv_leaf) - min_b[a] + 1;
    }
    if (i == 0) {                                    // PCL: "Leaf size is too small for the input dataset. Integer indices would overflow."
        const long long dx = (long long)((ordered_int_f32(box[3]) - ordered_int_f32(box[0])) * inv_leaf) + 1;
        const long long dy = (long long)((ordered_int_f32(box[4]) - ordered_int_f32(box[1])) * inv_leaf) + 1;
        const long long dz = (long long)((ordered_int_f32(box[5]) - ordered_int_f32(box[2])) * inv_leaf) + 1;
        if ((double)dx * (double)dy * (double)dz > 2147483647.0) *status = 1;
    }
    const int i0 = (int)(floorf(xyz[3 * (size_t)i] * inv_leaf) - (float)min_b[0]);
    const int i1 = (int)(floorf(xyz[3 * (size_t)i + 1] * inv_leaf) - (float)min_b[1]);
    const int i2 = (int)(floorf(xyz[3 * (size_t)i + 2] * inv_leaf) - (float)min_b[2]);
    keys[i] = (unsigned)(i0 + i1 * div_b[0] + i2 * div_b[0] * div_b[1]);
    vals[i] = i;
}
__global__ void k_vg_heads(const unsigned* __restrict__ keys_sorted, int n, int* __restrict__ head) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) head[i] = (i == 0 || keys_sorted[i] != keys_sorted[i - 1]) ? 1 : 0;
}
__global__ void k_vg_centroids(const float* __restrict__ xyz, const unsigned* __restrict__ keys_sorted, const int* __restrict__ vals_sorted,
                               const int* __restrict__ head, const int* __restrict__ rank, int n, float* __restrict__ out, int* __restrict__ count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (i == n - 1) *count = rank[i] + head[i];
    if (!head[i]) return;
    const unsigned k = keys_sorted[i];
    float sx = 0.f, sy = 0.f, sz = 0.f;
    int c = 0;
    for (int j = i; j < n && keys_sorted[j] == k; ++j) {
        const float* p = xyz + 3 * (size_t)vals_sorted[j];
        sx += p[0]; sy += p[1]; sz += p[2];
        ++c;
    }
    const float fc = (float)c;
    float* o = out + 3 * (size_t)rank[i];
    o[0] = sx / fc; o[1] = sy / fc; o[2] = sz / fc;
}

// ---------------------------------------------------------------------------------------
// scan preparation: Morton order in the BODY frame.  A rigid transform preserves spatial
// neighbourhoods, so the lanes of a warp query neighbouring map cells at every pose: similar trip
// counts (less divergence) and shared cache lines.  w carries the original scan index.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned morton_spread10(unsigned v) {
    v &= 0x3ffu;
    v = (v | (v << 16)) & 0x030000ffu;
    v = (v | (v << 8)) & 0x0300f00fu;
    v = (v | (v << 4)) & 0x030c30c3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}

__global__ void k_scan_keys(const float* __restrict__ xyz, int N, float ox, float oy, float oz, float inv_cell,
                            unsigned* __restrict__ keys, int* __restrict__ vals) {
    // 24-bit Morton key (8 bits per axis, clamped): the order only has to make the lanes of a warp neighbours;
    // three 8-bit radix passes instead of four shorten the upload's dependent kernel chain.
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const unsigned cx = (unsigned)fminf(fmaxf((xyz[3 * (size_t)i] - ox) * inv_cell, 0.f), 255.f);
    const unsigned cy = (unsigned)fminf(fmaxf((xyz[3 * (size_t)i + 1] - oy) * inv_cell, 0.f), 255.f);
    const unsigned cz = (unsigned)fminf(fmaxf((xyz[3 * (size_t)i + 2] - oz) * inv_cell, 0.f), 255.f);
    keys[i] = morton_spread10(cx) | (morton_spread10(cy) << 1) | (morton_spread10(cz) << 2);
    vals[i] = i;
}

__global__ void k_scan_gather(const float* __restrict__ xyz, int N, const int* __restrict__ vals_sorted,
                              float4* __restrict__ scan) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int src = vals_sorted[i];
    scan[i] = make_float4(xyz[3 * (size_t)src], xyz[3 * (size_t)src + 1], xyz[3 * (size_t)src + 2], __int_as_float(src));
}

// State in / result out as ONE launch each, reading / writing the page-locked host buffer directly (mapped memory):
// k_state_install replaces a host-to-device copy + a device-to-device copy (state pair + its saved copy),
// k_pack_result four small device-to-host copies -- on a 200 us frame every queued operation is 2-3 us of stream time.
__global__ void __launch_bounds__(256) k_state_install(const double* __restrict__ host_pair, State18* __restrict__ states) {
    constexpr int n = (int)(2 * sizeof(State18) / sizeof(double));
    double* d0 = reinterpret_cast<double*>(&states[0]);
    double* d3 = reinterpret_cast<double*>(&states[3]);
    for (int e = threadIdx.x; e < n; e += 256) {
        const double v = host_pair[e];
        d0[e] = v;
        d3[e] = v;
    }
}
__global__ void __launch_bounds__(256) k_pack_result(const State18* __restrict__ x, const unsigned* __restrict__ lio_ctrl, int lio_words,
                                                     const unsigned* __restrict__ vio_ctrl, int vio_words,
                                                     const unsigned* __restrict__ barrier, int bar_words, unsigned* __restrict__ host_out) {
    constexpr int nx = (int)(sizeof(State18) / sizeof(unsigned));
    const unsigned* xs = reinterpret_cast<const unsigned*>(x);
    for (int e = threadIdx.x; e < nx; e += 256) host_out[e] = xs[e];
    for (int e = threadIdx.x; e < lio_words; e += 256) host_out[nx + e] = lio_ctrl[e];
    for (int e = threadIdx.x; e < vio_words; e += 256) host_out[nx + lio_words + e] = vio_ctrl[e];
    for (int e = threadIdx.x; e < bar_words; e += 256) host_out[nx + lio_words + vio_words + e] = barrier[e];
}

// The whole upload ordering (keys, stable sort, gather, flag reset) in ONE block, for scans of up to BLOCK * ITEMS
// points: the per-frame persistent kernels leave one SM free (flb_capi.cu, `pers_cap`), and this kernel -- launched on
// the handle's scan stream -- orders frame k+1's scan on that SM while frame k's VIO update still runs on the other 147.
// Same keys and same tie order (stable, by input index) as k_scan_keys + the device-wide radix sort + k_scan_gather.
// Layout: item j of thread t is input index t * ITEMS + j ("blocked"; ITEMS odd so that the shared-memory transpose
// below is conflict-free); the sort's last pass leaves the output "striped" (position j * BLOCK + t), so the 16-byte
// stores are coalesced.
template <int kScanSortBlock, int ITEMS>
__global__ void __launch_bounds__(kScanSortBlock) k_scan_sort_block(const float* __restrict__ xyz, int N, float ox, float oy, float oz,
                                                                    float inv_cell, float4* __restrict__ scan,
                                                                    unsigned char* __restrict__ sel, unsigned char* __restrict__ plane_ok) {
    using Sort = cub::BlockRadixSort<unsigned, kScanSortBlock, ITEMS, int, 6>;
    extern __shared__ __align__(16) unsigned char s_sort[];
    unsigned* s_keys = reinterpret_cast<unsigned*>(s_sort);                       // dead before the sort reuses the bytes
    typename Sort::TempStorage& tmp = *reinterpret_cast<typename Sort::TempStorage*>(s_sort);
    const int t = threadIdx.x;
    // keys with coalesced reads, transposed through shared memory into the blocked arrangement
#pragma unroll 4
    for (int j = 0; j < ITEMS; ++j) {
        const int i = j * kScanSortBlock + t;
        unsigned key = 0x00FFFFFFu;                                               // padding: sorts last (stable: after real ties)
        if (i < N) {
            const unsigned cx = (unsigned)fminf(fmaxf((xyz[3 * (size_t)i] - ox) * inv_cell, 0.f), 255.f);
            const unsigned cy = (unsigned)fminf(fmaxf((xyz[3 * (size_t)i + 1] - oy) * inv_cell, 0.f), 255.f);
            const unsigned cz = (unsigned)fminf(fmaxf((xyz[3 * (size_t)i + 2] - oz) * inv_cell, 0.f), 255.f);
            key = morton_spread10(cx) | (morton_spread10(cy) << 1) | (morton_spread10(cz) << 2);
        }
        s_keys[i] = key;
    }
    __syncthreads();
    unsigned keys[ITEMS];
    int vals[ITEMS];
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        keys[j] = s_keys[t * ITEMS + j];
        vals[j] = t * ITEMS + j;
    }
    __syncthreads();
    Sort(tmp).SortBlockedToStriped(keys, vals, 0, 24);
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        const int pos = j * kScanSortBlock + t;
        if (pos < N) {
            const int src = vals[j];
            scan[pos] = make_float4(xyz[3 * (size_t)src], xyz[3 * (size_t)src + 1], xyz[3 * (size_t)src + 2], __int_as_float(src));
            sel[pos] = 1;               // point_selected_surf.resize(N, true) (src/laserMapping.cpp:1469)
            plane_ok[pos] = 0;
        }
    }
}

// ---------------------------------------------------------------------------------------
// standalone kNN (flb_knn): thread per query
// ---------------------------------------------------------------------------------------
__global__ void k_knn(GridDesc g, const int* __restrict__ cell_start, const float4* __restrict__ pts,
                      const float* __restrict__ q, int nq, int* __restrict__ idx, float* __restrict__ d2) {
    __shared__ int s_rows[18][128];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    Top5 t;
    knn5_grid(g, cell_start, pts, q[3 * (size_t)i], q[3 * (size_t)i + 1], q[3 * (size_t)i + 2], t, &s_rows[0][threadIdx.x], 128);
#pragma unroll
    for (int j = 0; j < kMatch; ++j) {
        const bool ok = (t.i[j] >= 0) && !(t.d[j] > g.max_d2);
        idx[(size_t)i * kMatch + j] = ok ? __float_as_int(__ldg(pts + t.i[j]).w) : -1;
        d2[(size_t)i * kMatch + j] = ok ? t.d[j] : INFINITY;
    }
}

// ---------------------------------------------------------------------------------------
// LIO pass
// ---------------------------------------------------------------------------------------
struct LioArgs {
    // inputs
    const float4* scan;          // N body points in Morton order, w = original index
    int N;
    GridDesc grid;
    const int* cell_start;
    const float4* map_pts;
    const State18* state;        // device state (pose read each pass)
    LioParamsDev prm;
    float plane_thr;
    // control: force_rematch < 0 -> read ctrl->nearest_search_en / ctrl->stop
    LioCtrl* ctrl;
    int force_rematch;
    const double* pose_override; // optional 12 doubles (R,p) on device; used by flb_lio_pass
    // per-point persistent (indexed by sorted position)
    unsigned char* sel;          // point_selected_surf
    float4* plane;               // cached pabcd
    unsigned char* plane_ok;
    // outputs
    double* partials;            // gridDim.x * lio_packed(W)
    // export, indexed by ORIGINAL scan index (may be null)
    float* x_world;              // N*3
    int* x_nn_idx;               // N*5
    float* x_nn_d2;              // N*5
    float* x_pabcd;              // N*4
    float* x_pd2;                // N
    unsigned char* x_rowmask;    // N
    double* x_rows;              // N*W
    double* x_meas;              // N
    unsigned long long* probe;   // profiling aid: stage timestamps of one thread (or null)
    int chunk;                   // persistent kernel: points per warp-chunk (1..32)
    int M;                       // map points (for the L2 prefetch)
    int prefetch;                // persistent kernel: stream the map + cell table into L2 before the first pass
    WarmList warm;               // persistent kernel: pages to touch before the first pass (n = 0: none)
};

template <int W>
__device__ __forceinline__ void lio_point(const LioArgs& a, const LioPose& pose, bool rematch, int i, bool& active,
                                          double (&row)[W], double& z, double& absres, int* rows, int rstride) {
    active = false;
    z = 0.0;
    absres = 0.0;
    const float4 b4 = __ldg(a.scan + i);
    const float pb[3] = {b4.x, b4.y, b4.z};
    const int oi = __float_as_int(b4.w);
    double pI[3];
    float pw[3];
    lio_body_to_world(pose, pb, pI, pw);
    bool sel;
    bool pok;
    float pabcd[4];
    const bool probe = a.probe && i == a.N / 2;
    if (probe) a.probe[0] = global_ns();
    if (rematch) {
        Top5 t;
        knn5_grid(a.grid, a.cell_start, a.map_pts, pw[0], pw[1], pw[2], t, rows, rstride);
        if (probe) a.probe[1] = global_ns();
        const bool five = t.i[kMatch - 1] >= 0;
        sel = five && !(t.d[kMatch - 1] > a.grid.max_d2);     // src/laserMapping.cpp:1549 (+ :1567 size check)
        pok = false;
        float nb[kMatch][3];
        int oidx[kMatch];
#pragma unroll
        for (int j = 0; j < kMatch; ++j) {
            oidx[j] = -1;
            if (t.i[j] >= 0) {
                const float4 P = __ldg(a.map_pts + t.i[j]);
                nb[j][0] = P.x; nb[j][1] = P.y; nb[j][2] = P.z;
                oidx[j] = __float_as_int(P.w);
            } else {
                nb[j][0] = nb[j][1] = nb[j][2] = 0.f;
            }
        }
        pabcd[0] = pabcd[1] = pabcd[2] = pabcd[3] = 0.f;
        if (sel) pok = plane_fit5(nb, a.plane_thr, pabcd);     // :1571
        if (probe) a.probe[2] = global_ns();
        a.plane[i] = make_float4(pabcd[0], pabcd[1], pabcd[2], pabcd[3]);
        a.plane_ok[i] = pok ? 1 : 0;
        if (a.x_nn_idx) {
#pragma unroll
            for (int j = 0; j < kMatch; ++j) {
                const bool ok = (t.i[j] >= 0) && !(t.d[j] > a.grid.max_d2);
                a.x_nn_idx[(size_t)oi * kMatch + j] = ok ? oidx[j] : -1;
                a.x_nn_d2[(size_t)oi * kMatch + j] = ok ? t.d[j] : INFINITY;
            }
        }
    } else {
        sel = a.sel[i] != 0;
        pok = a.plane_ok[i] != 0;
        const float4 pl = a.plane[i];
        pabcd[0] = pl.x; pabcd[1] = pl.y; pabcd[2] = pl.z; pabcd[3] = pl.w;
    }
    float pd2 = 0.f;
    if (sel) {
        sel = false;                                           // :1570
        if (pok) {
            if (lio_residual(pabcd, pw, pb, &pd2)) sel = true; // :1573-1584
        }
    }
    a.sel[i] = sel ? 1 : 0;
    active = sel && ((double)fabsf(pd2) <= 2.0);               // :1593
    if (active) {
        if (W == 6) lio_row6(pose, pI, pabcd, row);
        else lio_row12(pose, pI, pb, pabcd, row);
        z = -(double)pd2;                                      // :1628
        absres = (double)fabsf(pd2);
    }
    if (probe) a.probe[3] = global_ns();
    if (a.x_world) {
        a.x_world[3 * (size_t)oi] = pw[0]; a.x_world[3 * (size_t)oi + 1] = pw[1]; a.x_world[3 * (size_t)oi + 2] = pw[2];
#pragma unroll
        for (int k = 0; k < 4; ++k) a.x_pabcd[4 * (size_t)oi + k] = pabcd[k];
        a.x_pd2[oi] = pd2;
        a.x_rowmask[oi] = active ? 1 : 0;
#pragma unroll
        for (int k = 0; k < W; ++k) a.x_rows[(size_t)oi * W + k] = active ? row[k] : 0.0;
        a.x_meas[oi] = z;
    }
}

// Pose of this pass.  `through_l2`: the state was written by another SM earlier in this launch.
__device__ __forceinline__ void lio_make_pose(const LioArgs& a, LioPose& pose, bool through_l2) {
    const double* R = a.pose_override ? a.pose_override : a.state->rot;
    const double* p = a.pose_override ? a.pose_override + 9 : a.state->pos;
    for (int i = 0; i < 9; ++i) { pose.R[i] = through_l2 ? __ldcg(R + i) : R[i]; pose.R_LI[i] = a.prm.R_LI[i]; }
    for (int i = 0; i < 3; ++i) { pose.p[i] = through_l2 ? __ldcg(p + i) : p[i]; pose.t_LI[i] = a.prm.t_LI[i]; }
    m3_T(pose.R, pose.Rt);
    m3_T(pose.R_LI, pose.RLIt);
}

// Block-level reduction of per-thread accumulators acc[K] -> partials[blockIdx.x][K]:
// warp shuffle tree, then the warps in fixed order.
template <int K, int BLOCK>
__device__ __forceinline__ void block_reduce_store(const double (&acc)[K], double (*s_acc)[K], double* partials) {
    constexpr int NW = BLOCK / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if constexpr (K <= 32) {
        const double v = warp_transpose_reduce<K>(acc);
        if (lane < K) s_acc[warp][lane] = v;
    } else {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const double v = warp_sum(acc[k]);
            if (lane == 0) s_acc[warp][k] = v;
        }
    }
    __syncthreads();
    for (int q = threadIdx.x; q < K; q += BLOCK) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) s += s_acc[w][q];
        partials[(size_t)blockIdx.x * K + q] = s;
    }
}

template <int W>
__device__ __forceinline__ void lio_accumulate(double (&acc)[lio_packed(W)], const double (&row)[W], double z, double absres) {
    int k = 0;
#pragma unroll
    for (int r = 0; r < W; ++r) {
#pragma unroll
        for (int c = r; c < W; ++c) { acc[k] = fma(row[r], row[c], acc[k]); ++k; }
    }
#pragma unroll
    for (int r = 0; r < W; ++r) { acc[k] = fma(row[r], z, acc[k]); ++k; }
    acc[k] += 1.0;
    acc[k + 1] += absres;
}

// kernel-per-pass: one thread per scan point
template <int W, int BLOCK>
__device__ __forceinline__ void lio_pass_body(const LioArgs& a) {
    constexpr int K = lio_packed(W);
    __shared__ LioPose s_pose;
    __shared__ double s_acc[BLOCK / 32][K];
    __shared__ int s_rows[18][BLOCK];
    int rematch;
    if (a.force_rematch >= 0) {
        rematch = a.force_rematch;
    } else {
        if (a.ctrl->stop) return;
        rematch = a.ctrl->nearest_search_en;
    }
    if (threadIdx.x == 0) lio_make_pose(a, s_pose, false);
    __syncthreads();
    const int i = blockIdx.x * BLOCK + threadIdx.x;
    double acc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = 0.0;
    if (i < a.N) {
        bool active;
        double row[W], z, absres;
        lio_point<W>(a, s_pose, rematch != 0, i, active, row, z, absres, &s_rows[0][threadIdx.x], BLOCK);
        if (active) lio_accumulate<W>(acc, row, z, absres);
    }
    block_reduce_store<K, BLOCK>(acc, s_acc, a.partials);
}
template <int W, int BLOCK>
__global__ void __launch_bounds__(BLOCK) k_lio_pass(LioArgs a) { lio_pass_body<W, BLOCK>(a); }

// Batched frames (SURVEY.md section 7 H2(iv)): blockIdx.y = frame; every frame has its own scan, state, control
// block and partial sums (args[frame]), all share the map.  The pass of B frames is ONE launch, so the grid is B times
// larger than a frame's and the kernel runs where its throughput, not its latency, is what is measured.
template <int W, int BLOCK>
__global__ void __launch_bounds__(BLOCK) k_lio_pass_batched(const LioArgs* __restrict__ args) {
    __shared__ LioArgs s_a;
    {
        const unsigned* src = reinterpret_cast<const unsigned*>(args + blockIdx.y);
        unsigned* dst = reinterpret_cast<unsigned*>(&s_a);
        for (int e = threadIdx.x; e < (int)(sizeof(LioArgs) / sizeof(unsigned)); e += BLOCK) dst[e] = src[e];
    }
    __syncthreads();
    if ((int)blockIdx.x * BLOCK >= s_a.N) return;
    lio_pass_body<W, BLOCK>(s_a);
}

__global__ void __launch_bounds__(32) k_reduce_only(const double* partials, int nblocks, int K, double* out) {
    for (int q = threadIdx.x; q < K; q += 32) {
        double s = 0.0;
        int b = 0;
        for (; b + 8 <= nblocks; b += 8) {
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = partials[(size_t)(b + u) * K + q];
#pragma unroll
            for (int u = 0; u < 8; ++u) s += v[u];
        }
        for (; b < nblocks; ++b) s += partials[(size_t)b * K + q];
        out[q] = s;
    }
}

// ---------------------------------------------------------------------------------------
// Multi-GPU mailbox types and LL-style unit stores / loads (protocol: see "Fused NVLink exchange" below)
// ---------------------------------------------------------------------------------------
constexpr int kP2PMaxWorld = 8;
constexpr int kP2PErrCap = 16384;        // per-rank patch shard capacity of the error gather
struct __align__(16) P2PLine { unsigned d0, f0, d1, f1; };
struct P2PMailbox {
    P2PLine sums[2][kP2PMaxWorld][32];                       // [parity][source rank][k]; k = 31: that rank's patch count
    unsigned long long errs[2][kP2PMaxWorld][kP2PErrCap];    // [parity][source rank][local patch] = {tag : float bits}
};
struct P2PArgs {
    int world, rank;
    P2PMailbox* mail[kP2PMaxWorld];      // mail[rank] is the local one; others are peer mappings
    unsigned long long* seq;             // device-resident exchange counter (same value on every rank)
};

__device__ __forceinline__ void ll_store_line(P2PLine* p, double v, unsigned tag) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(v);
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"((unsigned)u), "r"(tag),
                 "r"((unsigned)(u >> 32)), "r"(tag)
                 : "memory");
}
__device__ __forceinline__ bool ll_load_line(const P2PLine* p, unsigned tag, double& v) {
    unsigned a, b, c, d;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "l"(p) : "memory");
    v = __longlong_as_double((long long)(((unsigned long long)c << 32) | a));
    return b == tag && d == tag;
}
__device__ __forceinline__ void ll_store_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ll_load_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
constexpr unsigned long long kP2PSpinLimit = 6000000ull;    // ~ seconds of polling: ranks may start far apart

// Worker side: publish one patch error to every rank (own mailbox included).
__device__ __forceinline__ void p2p_push_error(const P2PArgs& pp, unsigned tag, int local_patch, float err) {
    const unsigned long long unit = ((unsigned long long)tag << 32) | (unsigned long long)__float_as_uint(err);
    const int par = (int)(tag & 1u);
    for (int r = 0; r < pp.world; ++r) ll_store_u64(&pp.mail[r]->errs[par][pp.rank][local_patch], unit);
}

// ---------------------------------------------------------------------------------------
// VIO pass body: warp per patch, 2 pixels per lane
// ---------------------------------------------------------------------------------------
struct VioArgs {
    const unsigned char* img;    // continuous, stride == width
    CamModel cam;
    const double* pos;           // Pn*3
    const float* patch;          // Pn*192
    const int* search_level;     // Pn
    int Pn;
    const State18* state;
    const double* pose_override; // 12 doubles or null
    VioParamsDev prm;
    VioCtrl* ctrl;
    int force_level;             // >= 0 : use this level and ignore ctrl
    float* errors;               // 2 x err_stride (sub_sparse_map->errors; successive passes of the persistent
    int err_stride;              // kernel alternate between the halves, the kernel-per-pass path uses the first)
    double* partials;            // gridDim.x * kVioPacked
    double* x_z;                 // Pn*64 or null
    double* x_H;                 // Pn*64*6 or null
    P2PArgs p2p;                 // world > 1 (persistent kernel only): per-patch errors are pushed to every rank
    WarmList warm;               // persistent kernel: pages to touch before the first pass (n = 0: none)
    const int* Pn_dev;           // persistent kernel: when non-null the patch count is read from the device (the patch
                                 // list was built there by the visual-map selection, flb_vmap_select) and Pn is its capacity
    unsigned long long* err_units;   // persistent kernel, single GPU: 2 x err_stride self-validating {tag : error} units the leader
                                     // polls (the per-patch error of a warp's last patch is formed AFTER the block has arrived)
};

struct LatView {
    const float* p;
    __device__ __forceinline__ float operator()(int r, int c) const { return p[r * 11 + c]; }
};

// Per-warp inputs of one patch that do not depend on the pose: fetched once per launch when every
// warp owns a single patch (the persistent kernel), otherwise once per pass.
struct PatchIn {
    double pos[3];
    int search_level;
    float ref[3][2];          // reference patch values of this lane's two pixels, per pyramid level
};
__device__ __forceinline__ void vio_patch_load(const VioArgs& a, int i, int lane, PatchIn& in) {
    in.pos[0] = a.pos[3 * (size_t)i]; in.pos[1] = a.pos[3 * (size_t)i + 1]; in.pos[2] = a.pos[3 * (size_t)i + 2];
    in.search_level = a.search_level[i];
    const int x = lane >> 2, y0 = (lane & 3) * 2;
#pragma unroll
    for (int l = 0; l < 3; ++l) {
        // P[patch_size_total*level + x*8 + y]
        const float2 v = __ldg(reinterpret_cast<const float2*>(a.patch + (size_t)i * 192 + 64 * l + x * 8 + y0));
        in.ref[l][0] = v.x; in.ref[l][1] = v.y;
    }
}

// (float)((double)pe + sq) for pe >= 0 held as a double, without the two conversions: round the
// double sum to 24 significant bits, ties to even, on its bit pattern.  Exact whenever the result
// is a normal float or zero (the caller checks the operands).
__device__ __forceinline__ double round_to_f32_precision(double d) {
    unsigned long long u = (unsigned long long)__double_as_longlong(d);
    u += 0x0FFFFFFFull + ((u >> 29) & 1ull);
    u &= ~0x1FFFFFFFull;
    return __longlong_as_double((long long)u);
}

// One patch by one warp.  The 21 + 6 sums of the patch are reduced across the warp right away: lane l < 27
// adds the patch total of sum l to `accv` (so only one double per lane is carried from patch to patch);
// lane 0 also counts n_meas / skipped.
// Publish one per-patch error: the plain buffer (sub_sparse_map->errors), and -- persistent kernel -- the self-validating
// unit the leader(s) poll: every rank's mailbox in the fused multi-GPU mode, the local unit array otherwise.
__device__ __forceinline__ void vio_publish_error(const VioArgs& a, int i, float pe, unsigned p2p_tag, unsigned utag, int err_buf) {
    a.errors[(size_t)err_buf * a.err_stride + i] = pe;                            // :851
    if (p2p_tag) p2p_push_error(a.p2p, p2p_tag, i, pe);
    else if (utag) ll_store_u64(a.err_units + (size_t)err_buf * a.err_stride + i, ((unsigned long long)utag << 32) | (unsigned long long)__float_as_uint(pe));
}

// patch_error += res*res over the 64 pixels: float accumulator, double addend (:843) -- sequential, exact.  Lane 0.
__device__ __forceinline__ void vio_patch_error(const VioArgs& a, int i, const double* s_res, bool tiny, unsigned p2p_tag, unsigned utag,
                                                int err_buf, unsigned long long* wdbg) {
    if ((threadIdx.x & 31) == 0) {
        double ped = 0.0;
#pragma unroll 8
        for (int e = 0; e < 64; ++e) ped = round_to_f32_precision(ped + s_res[e]);
        float pe = (float)ped;
        if (tiny || !(ped < 3.0e38)) {                          // outside the shortcut's domain: literal form
            pe = 0.0f;
            for (int e = 0; e < 64; ++e) pe = (float)((double)pe + s_res[e]);
        }
        vio_publish_error(a, i, pe, p2p_tag, utag, err_buf);
        if (wdbg) wdbg[3] = global_ns();
    }
}

// `defer` (persistent kernel, last patch of this warp in the pass): the per-patch error chain is NOT run here; the caller
// runs vio_patch_error after its block has arrived at the pass barrier -- the chain (64 dependent steps by one lane,
// ~1.3 us) feeds only the leader's error sum, which is off the critical path, while the barrier is on it.  Returns true
// when a chain is pending (`tiny_out` is its argument; s_res must stay untouched until then).
__device__ __forceinline__ bool vio_patch(const VioArgs& a, const VioPose& pose, int level, int i, const PatchIn& in,
                                          float* s_lat, double* s_res, double& accv, double& n_meas, double& skipped,
                                          unsigned long long* wdbg = nullptr, unsigned p2p_tag = 0u, int err_buf = 0,
                                          unsigned utag = 0u, bool defer = false, bool* tiny_out = nullptr) {
    const int lane = threadIdx.x & 31;
    double acc[27];
#pragma unroll
    for (int k = 0; k < 27; ++k) acc[k] = 0.0;
    PatchGeom g;
    vio_patch_geom(a.cam, pose, in.pos, level, in.search_level, g);
    if (wdbg && lane == 0) wdbg[0] = global_ns();
    if (g.valid) {
        // stage the 11x11 tap lattice (stride = scale px) as float
        const int W = a.cam.width;
        {
            const unsigned char* base = a.img + (size_t)(g.v_i - 5 * g.scale) * W + (g.u_i - 5 * g.scale);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int e = lane + 32 * q;
                if (e < 121) {
                    const int r = e / 11, c = e - r * 11;
                    s_lat[e] = (float)__ldg(base + (size_t)r * g.scale * W + c * g.scale);
                }
            }
        }
        __syncwarp();
        if (wdbg && lane == 0) wdbg[1] = global_ns();
        LatView L{s_lat};
        const int x = lane >> 2, y0 = (lane & 3) * 2;
        // both pixels of this lane first (the patch geometry is dead afterwards), then the 21 + 6 products
        double row0[6], row1[6], res0, res1;
        vio_pixel(L, g, pose, x, y0, (level == 0) ? in.ref[0][0] : ((level == 1) ? in.ref[1][0] : in.ref[2][0]), row0, &res0);
        vio_pixel(L, g, pose, x, y0 + 1, (level == 0) ? in.ref[0][1] : ((level == 1) ? in.ref[1][1] : in.ref[2][1]), row1, &res1);
        const double sq0 = res0 * res0, sq1 = res1 * res1;
        s_res[x * 8 + y0] = sq0;
        s_res[x * 8 + y0 + 1] = sq1;
        bool tiny = (sq0 != 0.0 && !(sq0 >= 1.1754943508222875e-38)) || (sq1 != 0.0 && !(sq1 >= 1.1754943508222875e-38));
        // H^T H / H^T z partial sums: fused multiply-adds (the summation order over pixels, warps and
        // blocks already differs from the reference's dense product; parity is to tolerance here)
        {
            int k = 0;
#pragma unroll
            for (int r = 0; r < 6; ++r) {
#pragma unroll
                for (int c = r; c < 6; ++c) { acc[k] = fma(row1[r], row1[c], row0[r] * row0[c]); ++k; }
            }
#pragma unroll
            for (int r = 0; r < 6; ++r) acc[21 + r] = fma(row1[r], res1, row0[r] * res0);
        }
        if (a.x_z) {
            a.x_z[(size_t)i * 64 + x * 8 + y0] = res0;
            a.x_z[(size_t)i * 64 + x * 8 + y0 + 1] = res1;
#pragma unroll
            for (int r = 0; r < 6; ++r) {
                a.x_H[((size_t)i * 64 + x * 8 + y0) * 6 + r] = row0[r];
                a.x_H[((size_t)i * 64 + x * 8 + y0 + 1) * 6 + r] = row1[r];
            }
        }
        tiny = __any_sync(0xffffffffu, tiny);
        __syncwarp();
        if (wdbg && lane == 0) wdbg[2] = global_ns();
        if (lane == 0) n_meas += 64.0;
        if (defer) *tiny_out = tiny;
        else vio_patch_error(a, i, s_res, tiny, p2p_tag, utag, err_buf, wdbg);
        __syncwarp();
        accv += warp_transpose_reduce<27>(acc);
        return defer;
    } else {
        if (lane == 0) {
            skipped += 1.0;
            vio_publish_error(a, i, 0.0f, p2p_tag, utag, err_buf);
        }
        if (a.x_z) {
            for (int e = lane; e < 64; e += 32) {
                a.x_z[(size_t)i * 64 + e] = 0.0;
                for (int r = 0; r < 6; ++r) a.x_H[((size_t)i * 64 + e) * 6 + r] = 0.0;
            }
        }
    }
    return false;
}

__device__ __forceinline__ void vio_make_pose_from(const VioArgs& a, VioPose& pose, bool through_l2) {
    const double* Rg = a.pose_override ? a.pose_override : a.state->rot;
    const double* pg = a.pose_override ? a.pose_override + 9 : a.state->pos;
    double R[9], p[3];
    for (int i = 0; i < 9; ++i) R[i] = through_l2 ? __ldcg(Rg + i) : Rg[i];
    for (int i = 0; i < 3; ++i) p[i] = through_l2 ? __ldcg(pg + i) : pg[i];
    vio_make_pose(a.prm.Rci, a.prm.Pci, a.prm.Jdphi_dR, a.prm.Jdp_dR, R, p, pose);
}

template <int BLOCK>
__device__ __forceinline__ void vio_block_reduce_store(double accv, double n_meas, double skipped,
                                                       double (*s_acc)[kVioPacked], double* partials) {
    constexpr int NW = BLOCK / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane < 27) s_acc[warp][lane] = accv;
    if (lane == 0) { s_acc[warp][27] = n_meas; s_acc[warp][28] = skipped; }   // only lane 0 counts patches
    __syncthreads();
    for (int q = threadIdx.x; q < kVioPacked; q += BLOCK) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) s += s_acc[w][q];
        partials[(size_t)blockIdx.x * kVioPacked + q] = s;
    }
}

template <int BLOCK>
__device__ __forceinline__ void vio_pass_body(const VioArgs& a) {
    constexpr int NW = BLOCK / 32;
    __shared__ VioPose s_pose;
    __shared__ float s_lat[NW][128];
    __shared__ double s_res[NW][64];
    __shared__ double s_acc[NW][kVioPacked];
    int level;
    if (a.force_level >= 0) {
        level = a.force_level;
    } else {
        if (a.ctrl->stop) return;
        level = a.ctrl->level;
    }
    if (threadIdx.x == 0) vio_make_pose_from(a, s_pose, false);
    __syncthreads();
    const int warp = threadIdx.x >> 5;
    const int i = blockIdx.x * NW + warp;
    double accv = 0.0, n_meas = 0.0, skipped = 0.0;
    if (i < a.Pn) {
        PatchIn in;
        vio_patch_load(a, i, threadIdx.x & 31, in);
        vio_patch(a, s_pose, level, i, in, s_lat[warp], s_res[warp], accv, n_meas, skipped);
    }
    vio_block_reduce_store<BLOCK>(accv, n_meas, skipped, s_acc, a.partials);
}
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) k_vio_pass(VioArgs a) { vio_pass_body<BLOCK>(a); }

template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) k_vio_pass_batched(const VioArgs* __restrict__ args) {
    __shared__ VioArgs s_a;
    {
        const unsigned* src = reinterpret_cast<const unsigned*>(args + blockIdx.y);
        unsigned* dst = reinterpret_cast<unsigned*>(&s_a);
        for (int e = threadIdx.x; e < (int)(sizeof(VioArgs) / sizeof(unsigned)); e += BLOCK) dst[e] = src[e];
    }
    __syncthreads();
    vio_pass_body<BLOCK>(s_a);
}

// =======================================================================================
// Leader: reduction + the shared 18-DoF iterated-EKF step
// =======================================================================================
// Reference form (src/laserMapping.cpp:1664-1672, src/lidar_selection.cpp:871-878):
//     K1 = (H_T_H + (P/sigma)^-1)^-1,  H_T_H non-zero only in its leading 6x6 block
//     G[:, :6] = K1[:, :6] * HTH6 ;  sol = sign * K1[:, :6] * HTz + vec - G[:, :6] * vec[:6]
// Only K1[:, :6] is ever used.  By the block-inverse (Schur complement) identities, with
// P = [[P11, P12], [P21, P22]] (P11 the 6x6 rot/pos block):
//     K1[:6, :6] = (HTH6 + sigma * P11^-1)^-1 =: Kt        K1[6:, :6] = (P21 * P11^-1) * Kt
// so the two 18x18 inversions per pass become ONE 6x6 inversion per pass plus, once per update
// (the covariance only changes on the stopping pass), P11^-1 and B = P21 * P11^-1.  Identical in
// exact arithmetic; agrees with the partial-pivot-LU form to ~1e-12 relative.
struct PriorBlock {           // once per update, kept in global memory for later leaders
    double P11inv[36];
    double B[72];             // 12 x 6
};

struct LeaderSmem {
    State18 x, xp;            // L2 copies of state / prior
    double S[6 * 13];         // 6 x 12 Gauss-Jordan workspace, row stride 13 (odd: conflict-free)
    PriorBlock prior;
    double HTH[36], HTz[6];
    double K[kDim * 6];       // K1[:, :6]
    double vec[kDim], sol[kDim], Gc[kDim * 6];
    double xold[24];          // VIO: the pose/bias block before the accepted step (old_state, :863)
    double xspec[24];         // VIO: state (+) solution, formed before the accept test is known
    double top[6 * kDim];
    double packed[32];
    double part[16][32];
    int flags[8];             // [0] accept [1] docov [2] newlevel [3] singular [4] speculated [5] mispredicted
    float error;
    VioCtrl cspec;            // VIO: the control block of the speculated next pass
    int p2p_cnt[8];           // VIO: per-rank patch counts of this pass (kP2PMaxWorld)
};

// The 24 leading doubles (rot, pos, vel, bg, ba, grav) of x and xp: one L2 round trip for both.
__device__ __forceinline__ void load_poses_l2(State18* x, const State18* xg, State18* xp, const State18* xpg, int tid) {
    if (tid < 24) reinterpret_cast<double*>(x)[tid] = __ldcg(reinterpret_cast<const double*>(xg) + tid);
    else if (tid < 48) reinterpret_cast<double*>(xp)[tid - 24] = __ldcg(reinterpret_cast<const double*>(xpg) + tid - 24);
}
// The covariance only (needed for the prior block on the first pass and for the update on the last).
template <int NT>
__device__ __forceinline__ void load_cov_l2(State18* dst, const State18* src, int tid) {
    constexpr int PER = (kDim * kDim + NT - 1) / NT;
    double v[PER];
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int e = tid + u * NT;
        v[u] = (e < kDim * kDim) ? __ldcg(src->cov + e) : 0.0;
    }
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int e = tid + u * NT;
        if (e < kDim * kDim) dst->cov[e] = v[u];
    }
}
__device__ __forceinline__ void store_state(State18* dst, const State18* src, int tid, int nt, bool with_cov) {
    const double* s = reinterpret_cast<const double*>(src);
    double* d = reinterpret_cast<double*>(dst);
    const int n = with_cov ? (int)(sizeof(State18) / sizeof(double)) : 24;
    for (int e = tid; e < n; e += nt) d[e] = s[e];
}

// Fixed-order reduction of the block partials by a team of TN threads: its first TN/32-1 warps take one
// contiguous slice of the blocks each (summed in block order from batches of 16 independent L2 loads,
// guarded at the tail: adding +0.0 is exact), then the slices are combined left to right.  Meanwhile
// lane 0 of the team's LAST warp forms vec = state_propagat (-) state, which only needs sm.x / sm.xp.
template <int K, int TN, class TeamT>
__device__ __forceinline__ void team_reduce_vec(const double* partials, int nblocks, LeaderSmem& sm, int tid) {
    constexpr int PARTS = TN / 32 - 1;
    static_assert(PARTS >= 1 && PARTS <= 16 && K <= 32, "LeaderSmem::part is [16][32]");
    const int q = tid & 31, part = tid >> 5;
    if (part == PARTS) {
        if (q == 0) state_boxminus(sm.xp, sm.x, sm.vec);
    } else if (q < K) {
        const int per = (nblocks + PARTS - 1) / PARTS;
        const int b0 = part * per, b1 = min(nblocks, b0 + per);
        double s = 0.0;
        for (int b = b0; b < b1; b += 24) {       // 24 loads in flight: one round trip for a slice of up to 24 blocks
            double v[24];
#pragma unroll
            for (int u = 0; u < 24; ++u) v[u] = (b + u < b1) ? __ldcg(partials + (size_t)(b + u) * K + q) : 0.0;
#pragma unroll
            for (int u = 0; u < 24; ++u) s += v[u];
        }
        sm.part[part][q] = s;
    }
    TeamT::sync();
    if (tid < K) {
        double s = sm.part[0][tid];
#pragma unroll
        for (int p = 1; p < PARTS; ++p) s += sm.part[p][tid];
        sm.packed[tid] = s;
    }
    TeamT::sync();
}

// packed upper triangle (row-major, as accumulated by lio_accumulate / vio_patch) -> element (i, j)
__device__ __forceinline__ int sym6_index(int i, int j) {
    const int r = i < j ? i : j, c = i < j ? j : i;
    return r * 6 - (r * (r - 1)) / 2 + (c - r);
}

__device__ __forceinline__ void unpack_sym6(const double* packed, double* HTH, double* HTz) {
    int k = 0;
    for (int r = 0; r < 6; ++r)
        for (int c = r; c < 6; ++c) {
            HTH[r * 6 + c] = packed[k];
            HTH[c * 6 + r] = packed[k];
            ++k;
        }
    for (int r = 0; r < 6; ++r) HTz[r] = packed[k + r];
}

// The solve team: either the whole block (__syncthreads) or its first NT threads on named barrier 1,
// which leaves the remaining warp free to run something else concurrently (the VIO error sum).
template <int NT, bool NAMED>
struct Team {
    static constexpr int size = NT;
    static __device__ __forceinline__ void sync() {
        if (NAMED) asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");
        else __syncthreads();
    }
};

// Gauss-Jordan of the 6x12 system S (row stride 13) by threads 0..71 of the team (one element
// each), no pivoting (SPD).  A bad pivot raises sm_bad (shared flag).
template <class TeamT>
__device__ __forceinline__ void gj6(double* S, int* sm_bad, int tid) {
    const int i = tid / 12, j = tid - i * 12;
    for (int k = 0; k < 6; ++k) {
        double v = 0.0;
        if (tid < 72) {
            const double piv = S[k * 13 + k];
            if (!(fabs(piv) > 1e-300) || !isfinite(piv)) *sm_bad = 1;
            const double rkj = S[k * 13 + j] * __drcp_rn(piv);
            v = (i == k) ? rkj : S[i * 13 + j] - S[i * 13 + k] * rkj;
        }
        TeamT::sync();
        if (tid < 72) S[i * 13 + j] = v;
        TeamT::sync();
    }
}

// Once per update: P11^-1 and B = P21 * P11^-1 from sm.x.cov; stored to `out` (global) too.
template <class TeamT>
__device__ __forceinline__ void leader_prior(LeaderSmem& sm, PriorBlock* out, int tid) {
    if (tid < 72) {
        const int i = tid / 12, j = tid - i * 12;
        sm.S[i * 13 + j] = (j < 6) ? sm.x.cov[i * kDim + j] : ((j - 6 == i) ? 1.0 : 0.0);
    }
    TeamT::sync();
    gj6<TeamT>(sm.S, &sm.flags[3], tid);
    if (tid < 36) sm.prior.P11inv[tid] = sm.S[(tid / 6) * 13 + 6 + (tid % 6)];
    TeamT::sync();
    if (tid < 72) {
        const int i = tid / 6, j = tid - i * 6;   // B[i][j] = sum_k P[6+i][k] * P11inv[k][j]
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k) s += sm.x.cov[(6 + i) * kDim + k] * sm.prior.P11inv[k * 6 + j];
        sm.prior.B[tid] = s;
    }
    TeamT::sync();
    const double* src = reinterpret_cast<const double*>(&sm.prior);
    double* dst = reinterpret_cast<double*>(out);
    for (int e = tid; e < (int)(sizeof(PriorBlock) / sizeof(double)); e += TeamT::size) dst[e] = src[e];
}

// Later leaders: fetch the prior block (one double per thread, tid < 108) into a register early and
// commit it to shared memory once the reduction is done, so the L2 round trip hides behind it.
constexpr int kPriorDoubles = (int)(sizeof(PriorBlock) / sizeof(double));
__device__ __forceinline__ double prior_prefetch(const PriorBlock* in, int tid) {
    return (tid < kPriorDoubles) ? __ldcg(reinterpret_cast<const double*>(in) + tid) : 0.0;
}
__device__ __forceinline__ void prior_commit(LeaderSmem& sm, double v, int tid) {
    if (tid < kPriorDoubles) reinterpret_cast<double*>(&sm.prior)[tid] = v;
}

// The per-pass solve, by ONE warp, registers and shuffles only.  With K = K1[:, :6] = [Kt; B Kt]:
//     solution = sign K HTz + vec - (K HTH6) vec[:6] = vec + [y; B y],   y = Kt w,  w = sign HTz - HTH6 vec[:6]
// so a pass needs one 6x6 solve with a single right-hand side, not the gain itself (the gain is only
// formed for the covariance update, leader_gain below).  Lane j < 6 holds column j of
// A = HTH6 + sigma P11^-1, lanes >= 6 all hold the right-hand side; Gauss-Jordan without pivoting
// (SPD).  Requires sm.packed, sm.vec, sm.prior; writes sm.sol; a bad pivot raises sm.flags[3].
__device__ __forceinline__ void leader_fast_solve(LeaderSmem& sm, double sigma, double sign, int lane) {
    const unsigned full = 0xffffffffu;
    double col[6];
    if (lane < 6) {
#pragma unroll
        for (int i = 0; i < 6; ++i) col[i] = sm.packed[sym6_index(i, lane)] + sigma * sm.prior.P11inv[i * 6 + lane];
    } else {
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            double a = 0.0;
#pragma unroll
            for (int k = 0; k < 6; ++k) a += sm.packed[sym6_index(i, k)] * sm.vec[k];
            col[i] = sign * sm.packed[21 + i] - a;
        }
    }
    bool bad = false;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        double ck[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) ck[i] = __shfl_sync(full, col[i], k);
        const double piv = ck[k];
        bad = bad || !(fabs(piv) > 1e-300) || !isfinite(piv);
        const double r = col[k] * __drcp_rn(piv);
#pragma unroll
        for (int i = 0; i < 6; ++i) col[i] = (i == k) ? r : col[i] - ck[i] * r;
    }
    // lanes >= 6 now hold y
    if (lane >= 8 && lane < 8 + kDim) {
        const int idx = lane - 8;
        double v = sm.vec[idx];
        if (idx < 6) {
#pragma unroll
            for (int i = 0; i < 6; ++i) if (i == idx) v += col[i];
        } else {
            double a = 0.0;
#pragma unroll
            for (int k = 0; k < 6; ++k) a += sm.prior.B[(idx - 6) * 6 + k] * col[k];
            v += a;
        }
        sm.sol[idx] = v;
    }
    if (lane == 0 && bad) sm.flags[3] = 1;
    __syncwarp();
}

// The gain of a pass, needed only where the reference updates the covariance with it
// (src/laserMapping.cpp:1715, src/lidar_selection.cpp:980): Kt = (HTH6 + sigma P11^-1)^-1,
// K = [Kt; B Kt], Gc = K HTH6 (the non-zero columns of G).  Whole team; HTH6 = sm.HTH.
template <class TeamT>
__device__ __forceinline__ void leader_gain(LeaderSmem& sm, double sigma, int tid) {
    if (tid < 72) {
        const int i = tid / 12, j = tid - i * 12;
        sm.S[i * 13 + j] = (j < 6) ? sm.HTH[i * 6 + j] + sigma * sm.prior.P11inv[i * 6 + j] : ((j - 6 == i) ? 1.0 : 0.0);
    }
    TeamT::sync();
    gj6<TeamT>(sm.S, &sm.flags[3], tid);
    if (tid < 36) sm.K[tid] = sm.S[(tid / 6) * 13 + 6 + (tid % 6)];   // Kt
    TeamT::sync();
    if (tid < 72) {
        const int i = tid / 6, j = tid - i * 6;                       // Kb = B * Kt
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k) s += sm.prior.B[i * 6 + k] * sm.K[k * 6 + j];
        sm.K[36 + tid] = s;
    }
    TeamT::sync();
    if (tid < kDim * 6) {
        const int i = tid / 6, j = tid - i * 6;                       // Gc = K * HTH6
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k) s += sm.K[i * 6 + k] * sm.HTH[k * 6 + j];
        sm.Gc[tid] = s;
    }
    TeamT::sync();
}

// cov (smem state) <- cov - Gc * cov[:6,:]   ( == (I - G) * cov, G non-zero only in columns 0..5 )
__device__ __forceinline__ void leader_cov_update(LeaderSmem& sm, const double* Gc, int tid, int nt) {
    for (int e = tid; e < 6 * kDim; e += nt) sm.top[e] = sm.x.cov[e];
    __syncthreads();
    for (int e = tid; e < kDim * kDim; e += nt) {
        const int i = e / kDim, j = e - i * kDim;
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k) s += Gc[i * 6 + k] * sm.top[k * kDim + j];
        sm.x.cov[e] = sm.x.cov[e] - s;
    }
    __syncthreads();
}

// =======================================================================================
// Fused NVLink exchange (multi-GPU, SURVEY.md section 8e): no NCCL in the data path
// =======================================================================================
// Every rank owns a mailbox in its device memory; peers map it (CUDA IPC).  All traffic is "LL" style
// (NCCL's low-latency protocol): every unit a peer writes carries its own validity tag next to the payload,
// inside one store instruction whose 8-byte halves are atomic, so the reader polls the DATA -- there is no
// separate flag, no __threadfence_system, and one NVLink traversal per exchange:
//   * packed normal-equation sums: one 16-byte line {lo32, tag, hi32, tag} per double, written by the leader
//     block of each rank straight into every rank's mailbox (own included) and summed in rank order by
//     everyone: bit-identical sums everywhere, so the replicated solve yields bit-identical states;
//   * VIO per-patch float errors: one 8-byte unit {float bits, tag} per patch, pushed to every rank by the
//     WORKER warp that computed it, as soon as the patch is done (long before the pass ends); the leader's
//     error-sum warp stages them into shared memory in global patch order while it checks the tags.
// The tag is the exchange number (a device-resident counter that advances identically on every rank: one
// per pass).  Slots are double-buffered by tag parity: a rank can be at most one exchange ahead of the
// slowest one (it cannot finish exchange k+1 without that rank's k+1 contribution, which that rank only
// sends after it has consumed exchange k).
// All-reduce sm.packed[0..K) across ranks in rank order, executed by a team of threads (TeamT).  Uses sm.part as
// the receive staging.  (Line 31 of every rank's slot is the VIO patch count, pushed at the start of the pass.)
template <int K, class TeamT>
__device__ __forceinline__ void p2p_exchange(const P2PArgs& pp, LeaderSmem& sm, unsigned tag, int tid, int* timeout_flag) {
    static_assert(K <= 31, "line 31 is the patch count");
    const int par = (int)(tag & 1u);
    const int nline = pp.world * 32;
    for (int e = tid; e < nline; e += TeamT::size) {
        const int r = e >> 5, k = e & 31;
        if (k < K) ll_store_line(&pp.mail[r]->sums[par][pp.rank][k], sm.packed[k], tag);
    }
    for (int e = tid; e < nline; e += TeamT::size) {
        const int r = e >> 5, k = e & 31;
        if (k < K) {
            const P2PLine* src = &pp.mail[pp.rank]->sums[par][r][k];
            double v;
            unsigned long long spins = 0;
            while (!ll_load_line(src, tag, v)) {
                if (++spins > kP2PSpinLimit) { *timeout_flag = 1; break; }
            }
            sm.part[r][k] = v;
        }
    }
    TeamT::sync();
    if (tid < K) {
        double s = 0.0;
        for (int r = 0; r < pp.world; ++r) s += sm.part[r][tid];
        sm.packed[tid] = s;
    }
    TeamT::sync();
}

struct LioSolveArgs {
    State18* state;
    const State18* state_prop;
    LioCtrl* ctrl;
    PriorBlock* prior;
    const double* partials;  // nblocks * lio_packed(6)   (or 1 x packed after an all-reduce)
    int nblocks;
    LioParamsDev prm;
    P2PArgs p2p;             // world <= 1: single GPU
    int* timeout_flag;       // GridBarrier::timeout
    // persistent kernel: where the update STARTS from when that is not *state / *state_prop (a pending
    // flb_state_reset_enqueue: the saved pair).  The leader copies both into state / state_prop first.
    const State18* init_x;
    const State18* init_xp;
};

// Warp-level publication of the pose packet (see "Pose packet" below): 8-byte units {word, flag}.
constexpr int kPktUnits = 96;
constexpr int kStateWords = 48;                          // rot, pos, vel, bg, ba, grav as 32-bit words
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
template <int NC>
__device__ __forceinline__ void pkt_publish_warp(unsigned long long* pkt, const State18& x, const void* c, unsigned flag, int lane) {
    static_assert(kStateWords + NC <= kPktUnits, "packet too small");
    const unsigned* xs = reinterpret_cast<const unsigned*>(&x);
    const unsigned* cs = reinterpret_cast<const unsigned*>(c);
#pragma unroll
    for (int e = lane; e < kStateWords + NC; e += 32) {
        const unsigned w = (e < kStateWords) ? xs[e] : cs[e - kStateWords];
        st_relaxed_u64(pkt + e, ((unsigned long long)flag << 32) | w);
    }
}

// One LIO leader step (whole block, NT threads), in two halves.  Requires the 24 pose/bias doubles of
// sm.x and sm.xp and the control block `c` (shared memory) to be current; `first`: first pass of this update.
//   lio_leader_solve : reduce -> [exchange] -> warp 0: solve, state (+)= solution, loop control (c) and,
//                      in the persistent kernel (pkt != nullptr), publication of the new pose
//   lio_leader_finish: covariance update on the stopping pass; stores what later launches / the host need
#define FLB_STAMP(k) do { if (fine && threadIdx.x == 0) fine[k] = global_ns(); } while (0)
template <int NT>
__device__ __forceinline__ void lio_leader_solve(const LioSolveArgs& s, LeaderSmem& sm, LioCtrl& c, bool first,
                                                 unsigned long long* pkt, unsigned flag, int resident,
                                                 unsigned long long* fine = nullptr, unsigned p2p_tag = 0u) {
    constexpr int K = lio_packed(6);
    constexpr int NC = (int)(sizeof(LioCtrl) / sizeof(unsigned));
    using T = Team<NT, false>;
    const int tid = threadIdx.x;
    const int T_it = s.prm.max_iteration;
    // resident != 0 (persistent kernel): covariance and prior block already sit in this block's shared
    // memory (leader_prepare); resident == 2 flags a singular prior.  Otherwise the first leader forms the
    // prior block and later leaders fetch it while the partials are being reduced.
    if (first && !resident) load_cov_l2<NT>(&sm.x, s.state, tid);
    const double pri = (first || resident) ? 0.0 : prior_prefetch(s.prior, tid);
    if (tid == 0) sm.flags[3] = (resident == 2) ? 1 : 0;
    FLB_STAMP(0);
    team_reduce_vec<K, NT, T>(s.partials, s.nblocks, sm, tid);
    if (!first && !resident) prior_commit(sm, pri, tid);
    if (p2p_tag) p2p_exchange<K, T>(s.p2p, sm, p2p_tag, tid, s.timeout_flag);
    if (first && !resident) leader_prior<T>(sm, s.prior, tid);
    __syncthreads();
    FLB_STAMP(1);
    if (tid < 32) {
        leader_fast_solve(sm, s.prm.sigma, +1.0, tid);
        FLB_STAMP(2);
        if (tid == 0) {
            const bool ok = sm.flags[3] == 0;
            const int iterCount = c.iterCount, rematch_num = c.rematch_num, nearest = c.nearest_search_en;
            if (first) {
                c.passes = c.knn_passes = 0;
                c.rows_total = 0;
                c.status = 0;
            }
            const int n_eff = (int)sm.packed[K - 2];
            c.passes += 1;
            c.knn_passes += nearest ? 1 : 0;
            c.n_eff_last = n_eff;
            c.res_mean_last = sm.packed[K - 1] / (double)n_eff;                            // :1602
            c.rows_total += n_eff;
            state_boxplus(sm.x, sm.sol);                                                   // :1683
            bool converged = false;
            if ((norm3(sm.sol) * 57.3 < s.prm.conv_rot_deg) && (norm3(sm.sol + 3) * 100 < s.prm.conv_pos_cm))
                converged = true;                                                          // :1688
            int nn = 0, rn = rematch_num;
            if (converged || ((rn == 0) && (iterCount == (T_it - 2)))) { nn = 1; rn++; }    // :1700-1705
            int stop = 0;
            if (rn >= 2 || (iterCount == T_it - 1)) stop = 1;                               // :1708
            if (!ok) { stop = 1; c.status = -5; }
            c.converged_last = converged ? 1 : 0;
            c.iterCount = iterCount + 1;
            c.rematch_num = rn;
            c.nearest_search_en = nn;
            c.stop = stop;
            sm.flags[0] = stop;
            sm.flags[1] = ok ? 1 : 0;
        }
        __syncwarp();
        if (pkt) pkt_publish_warp<NC>(pkt, sm.x, &c, flag, tid);
    }
    __syncthreads();
    FLB_STAMP(3);
}

// `store_always`: kernel-per-pass path (state and control live in global memory between launches).
template <int NT>
__device__ __forceinline__ void lio_leader_finish(const LioSolveArgs& s, LeaderSmem& sm, const LioCtrl& c, bool first,
                                                  bool store_always, int resident, unsigned long long* fine = nullptr) {
    const int tid = threadIdx.x;
    const bool stop = sm.flags[0] != 0;
    const bool do_cov = stop && sm.flags[1];
    if (do_cov) {
        if (tid < 36) sm.HTH[tid] = sm.packed[sym6_index(tid / 6, tid % 6)];
        if (!first && !resident) load_cov_l2<NT>(&sm.x, s.state, tid);
        __syncthreads();
        leader_gain<Team<NT, false>>(sm, s.prm.sigma, tid);
        leader_cov_update(sm, sm.Gc, tid, NT);                                          // :1715
    }
    if (stop || store_always) {
        store_state(s.state, &sm.x, tid, NT, do_cov);
        if (tid == 0) *s.ctrl = c;
    }
    FLB_STAMP(4);
}

__global__ void __launch_bounds__(32) k_lio_begin(LioCtrl* ctrl) {
    if (threadIdx.x == 0) {
        LioCtrl c;
        c.iterCount = -1;
        c.rematch_num = 0;
        c.nearest_search_en = 1;
        c.stop = 0;
        c.passes = c.knn_passes = c.n_eff_last = c.converged_last = 0;
        c.status = 0;
        c.res_mean_last = 0.0;
        c.rows_total = 0;
        *ctrl = c;
    }
}

__device__ __forceinline__ void lio_finalize_body(const LioSolveArgs& s) {
    __shared__ LeaderSmem sm;
    __shared__ LioCtrl c;
    if (s.ctrl->stop) return;
    const int tid = threadIdx.x;
    if (tid == 0) c = *s.ctrl;
    load_poses_l2(&sm.x, s.state, &sm.xp, s.state_prop, tid);
    __syncthreads();
    const bool first = c.passes == 0;
    lio_leader_solve<kLeaderBlock>(s, sm, c, first, nullptr, 0u, 0);
    lio_leader_finish<kLeaderBlock>(s, sm, c, first, true, 0);
}
__global__ void __launch_bounds__(kLeaderBlock) k_lio_finalize(LioSolveArgs s) { lio_finalize_body(s); }
__global__ void __launch_bounds__(kLeaderBlock) k_lio_finalize_batched(const LioSolveArgs* __restrict__ args) {
    __shared__ LioSolveArgs s_s;
    {
        const unsigned* src = reinterpret_cast<const unsigned*>(args + blockIdx.x);
        unsigned* dst = reinterpret_cast<unsigned*>(&s_s);
        for (int e = threadIdx.x; e < (int)(sizeof(LioSolveArgs) / sizeof(unsigned)); e += kLeaderBlock) dst[e] = src[e];
    }
    __syncthreads();
    lio_finalize_body(s_s);
}
__global__ void k_lio_begin_batched(LioCtrl* const* ctrls, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    LioCtrl c;
    c.iterCount = -1; c.rematch_num = 0; c.nearest_search_en = 1; c.stop = 0;
    c.passes = c.knn_passes = c.n_eff_last = c.converged_last = 0; c.status = 0;
    c.res_mean_last = 0.0; c.rows_total = 0;
    *ctrls[b] = c;
}

struct VioSolveArgs {
    State18* state;
    const State18* state_prop;
    State18* old_state;
    VioCtrl* ctrl;
    PriorBlock* prior;
    double* G_last;          // 18x6, the G of the last accepted solve (:874, used at :980)
    const double* partials;
    int nblocks;
    const float* errors;     // all patches, patch order (local shard in the fused multi-GPU mode); two halves of
    int err_stride;          // err_stride floats, written alternately by successive passes of the persistent kernel
    int Pn_total;
    VioParamsDev prm;
    P2PArgs p2p;             // world <= 1: single GPU
    int* timeout_flag;
    int prior_from_state;    // persistent kernel: state_propagat = state (a pending flb_state_set_prior_enqueue, laserMapping.cpp:1292)
    const unsigned long long* err_units;   // see VioArgs::err_units (null: read `errors`)
};

constexpr int kErrChunk = 2048;          // staging capacity of the kernel-per-pass finalize kernel (static shared memory)
// threads of the leader block that gather + sum the per-patch errors: 160 of the persistent kernel's 512 (the other 352 reduce
// the 146 block partials in ten slices of 15: one round trip), 128 of the finalize kernel's 256
constexpr int kVioDbg = 8 + 4 * 16;   // debug stamps per block (tracing only)

// One VIO leader step (whole block, NT threads), in two halves like the LIO one.  Requires the 24
// pose/bias doubles of sm.x / sm.xp and the control block `c` (shared memory); c.level is the pyramid
// level of the pass just done.
template <int NT>
__device__ __forceinline__ void vio_leader_solve(const VioSolveArgs& s, LeaderSmem& sm, VioCtrl& c, float* s_err, bool first,
                                                 unsigned long long* pkt, unsigned flag, int resident,
                                                 unsigned long long* fine = nullptr, unsigned p2p_tag = 0u, int err_buf = 0,
                                                 int err_cap = kErrChunk, int pn_override = -1) {
    constexpr int NC = (int)(sizeof(VioCtrl) / sizeof(unsigned));
    const int tid = threadIdx.x;
    const int pn_total = pn_override >= 0 ? pn_override : s.Pn_total;
    const bool multi = p2p_tag != 0u;
    const int level = c.level;
    const float* errs_pass = s.errors + (size_t)err_buf * s.err_stride;     // this pass's half of the error buffer
    const int nsrc = multi ? s.p2p.world : 1;
    const int par = (int)(p2p_tag & 1u);
    // Per-patch errors of this pass, in global patch order (rank 0's shard, then rank 1's, ...: contiguous block
    // partition).  Single GPU: this rank's error buffer.  Fused multi-GPU mode: every rank's worker warps pushed
    // {error, tag} units into this rank's mailbox while the pass was running, and each rank's patch count came
    // with the first block of its pass (line 31); every unit is validated by its tag.
    constexpr int kErrTeam = NT >= 512 ? 160 : 128;
    static_assert(NT - kErrTeam >= kDim * 6 && NT - kErrTeam >= 64, "solve team too small");
    if (tid >= NT - kErrTeam) {
        // ---- error team (the last kErrTeam threads): gather, then its last warp sums
        const int et = tid - (NT - kErrTeam);
        if (multi) {
            if (et < nsrc) {
                double cnt = 0.0;
                unsigned long long spins = 0;
                while (!ll_load_line(&s.p2p.mail[s.p2p.rank]->sums[par][et][31], p2p_tag, cnt))
                    if (++spins > kP2PSpinLimit) { *s.timeout_flag = 1; cnt = 0.0; break; }
                sm.p2p_cnt[et] = (int)cnt;
            }
        } else if (et == 0) {
            sm.p2p_cnt[0] = pn_total;
        }
        asm volatile("bar.sync 4, %0;" ::"n"(kErrTeam) : "memory");
        int total = 0;
        for (int r = 0; r < nsrc; ++r) total += sm.p2p_cnt[r];
        const unsigned want_tag = multi ? p2p_tag : (flag | 0x80000000u);
        auto unit_of = [&](int e) -> const unsigned long long* {
            if (!multi) return s.err_units + (size_t)err_buf * s.err_stride + e;
            int r = 0;
            while (r + 1 < nsrc && e >= sm.p2p_cnt[r]) { e -= sm.p2p_cnt[r]; ++r; }
            return &s.p2p.mail[s.p2p.rank]->errs[par][r][e];
        };
        auto fetch = [&](int e) -> float {
            if (!multi && s.err_units == nullptr) return __ldcg(errs_pass + e);
            const unsigned long long* unit;
            if (multi) {
                int r = 0;
                while (r + 1 < nsrc && e >= sm.p2p_cnt[r]) { e -= sm.p2p_cnt[r]; ++r; }
                unit = &s.p2p.mail[s.p2p.rank]->errs[par][r][e];
            } else {
                unit = s.err_units + (size_t)err_buf * s.err_stride + e;
            }
            unsigned long long u = ll_load_u64(unit);
            unsigned long long spins = 0;
            while ((unsigned)(u >> 32) != want_tag) {
                if (++spins > kP2PSpinLimit) { *s.timeout_flag = 1; break; }
                u = ll_load_u64(unit);
            }
            return __uint_as_float((unsigned)u);
        };
        // Gather and sum are PIPELINED: all warps of the team but the last stage the errors into shared memory in slices
        // of kErrSlice (each thread 16 independent loads / unit polls per slice: one L2 round trip per attempt) and hand
        // each slice over through a named barrier (arrive / sync pairs, two ids alternating); lane 0 of the last warp runs
        // the exact sequential float sum (:852) behind them, one FADD latency per patch, 16 addends per step with the next
        // 16 already fetched from shared memory.  The chain is the longer of the two (2 k patches: 4 us, 10 k: 20 us), so
        // the gather costs one round trip, not one per slice.  Both are hidden behind the other threads' reduce + solve
        // and -- in the persistent kernel -- behind the next pass, which has already been started on the accept branch.
        constexpr int kStagers = kErrTeam - 32, kPer = 16, kErrSlice = kStagers * kPer;
        const int n0 = min(err_cap, total);
        const int nslices = (n0 + kErrSlice - 1) / kErrSlice;
        if (et < kStagers) {
            const bool units = multi || s.err_units != nullptr;
            for (int c = 0; c < nslices; ++c) {
                // a barrier id is reused every other slice: do not arrive for slice c before the chain warp has taken slice
                // c - 2 (EMPTY[c & 1]: the chain warp arrives, the stagers sync)
                if (c >= 2) {
                    if (c & 1) asm volatile("bar.sync 8, %0;" ::"n"(kErrTeam) : "memory");
                    else asm volatile("bar.sync 7, %0;" ::"n"(kErrTeam) : "memory");
                }
                const int b0 = c * kErrSlice + et;
                if (!units) {
                    // plain floats, complete when the blocks arrived: 16 independent loads
                    float v[kPer];
#pragma unroll
                    for (int u = 0; u < kPer; ++u) {
                        const int e = b0 + u * kStagers;
                        v[u] = (e < n0) ? __ldcg(errs_pass + e) : 0.f;
                    }
#pragma unroll
                    for (int u = 0; u < kPer; ++u) {
                        const int e = b0 + u * kStagers;
                        if (e < n0) s_err[e] = v[u];
                    }
                } else {
                    // self-validating units, still being written when the poll starts: all of this thread's units of the
                    // slice are polled together (one round trip per attempt for the lot), each re-polled until its tag is right
                    const unsigned long long* up[kPer];
                    unsigned pending = 0u;
#pragma unroll
                    for (int u = 0; u < kPer; ++u) {
                        const int e = b0 + u * kStagers;
                        up[u] = unit_of(e < n0 ? e : 0);
                        if (e < n0) pending |= 1u << u;
                    }
                    unsigned long long spins = 0;
                    while (pending) {
                        unsigned long long uv[kPer];
#pragma unroll
                        for (int u = 0; u < kPer; ++u) uv[u] = (pending >> u & 1u) ? ll_load_u64(up[u]) : 0ull;
#pragma unroll
                        for (int u = 0; u < kPer; ++u)
                            if ((pending >> u & 1u) && (unsigned)(uv[u] >> 32) == want_tag) {
                                s_err[b0 + u * kStagers] = __uint_as_float((unsigned)uv[u]);
                                pending &= ~(1u << u);
                            }
                        if (pending && ++spins > kP2PSpinLimit) { *s.timeout_flag = 1; break; }
                    }
                }
                // hand slice c to the chain warp: named barrier FULL[c & 1] (stagers arrive, the chain warp syncs)
                if (c & 1) asm volatile("bar.arrive 6, %0;" ::"n"(kErrTeam) : "memory");
                else asm volatile("bar.arrive 5, %0;" ::"n"(kErrTeam) : "memory");
            }
        } else {
        const int lane = et - kStagers;
        float e_run = 0.0f;
        {
            float e = 0.0f;
            for (int c = 0; c < nslices; ++c) {
                if (c & 1) asm volatile("bar.sync 6, %0;" ::"n"(kErrTeam) : "memory");
                else asm volatile("bar.sync 5, %0;" ::"n"(kErrTeam) : "memory");
                if (fine && c == 0 && lane == 0) fine[0] = global_ns();
                if (lane == 0) {
                    const int i0 = c * kErrSlice, i1 = min(i0 + kErrSlice, n0);
                    const float4* s4 = reinterpret_cast<const float4*>(s_err);
                    int i = i0;
                    if (i1 - i0 >= 16) {
                        float4 n0v = s4[i0 >> 2], n1v = s4[(i0 >> 2) + 1], n2v = s4[(i0 >> 2) + 2], n3v = s4[(i0 >> 2) + 3];
                        for (; i + 16 <= i1; i += 16) {
                            const float4 c0 = n0v, c1 = n1v, c2 = n2v, c3 = n3v;
                            {   // unconditional, index clamped into this slice (unused past its end)
                                const int q = min((i >> 2) + 4, (i1 >> 2) - 4);
                                n0v = s4[q]; n1v = s4[q + 1]; n2v = s4[q + 2]; n3v = s4[q + 3];
                            }
                            e = e + c0.x; e = e + c0.y; e = e + c0.z; e = e + c0.w;
                            e = e + c1.x; e = e + c1.y; e = e + c1.z; e = e + c1.w;
                            e = e + c2.x; e = e + c2.y; e = e + c2.z; e = e + c2.w;
                            e = e + c3.x; e = e + c3.y; e = e + c3.z; e = e + c3.w;
                        }
                    }
                    for (; i < i1; ++i) e = e + s_err[i];
                }
                __syncwarp();
                if (c + 2 < nslices) {
                    if (c & 1) asm volatile("bar.arrive 8, %0;" ::"n"(kErrTeam) : "memory");
                    else asm volatile("bar.arrive 7, %0;" ::"n"(kErrTeam) : "memory");
                }
            }
            e_run = e;
        }
        __syncwarp();
        // beyond the staged capacity (more patches than err_cap): this warp stages and sums the rest chunk by chunk
        for (int base = err_cap; base < total; base += err_cap) {
            const int nchunk = min(err_cap, total - base);
            e_run = __shfl_sync(0xffffffffu, e_run, 0);
            for (int e = lane; e < nchunk; e += 32) s_err[e] = fetch(base + e);
            __syncwarp();
            if (lane == 0) {
                float e = e_run;
                for (int i = 0; i < nchunk; ++i) e = e + s_err[i];
                e_run = e;
            }
            __syncwarp();
        }
        if (lane == 0) sm.error = e_run;
        if (fine && lane == 0) fine[3] = global_ns();
        asm volatile("bar.sync 3, 64;" ::: "memory");                       // hand the error to warp 0
        }
    } else {
        // Solve team (first NT-32 threads, named barrier 1).  The covariance is constant during ComputeJ
        // (only :980 changes it, on the last pass), so old_state carries the 24 pose/bias doubles only.
        using T = Team<NT - kErrTeam, true>;
        if (first && !resident) load_cov_l2<NT - kErrTeam>(&sm.x, s.state, tid);
        const double pri = (first || resident) ? 0.0 : prior_prefetch(s.prior, tid);
        if (first) store_state(s.old_state, &sm.x, tid, NT - kErrTeam, false);           // old_state = *state (:747)
        if (tid == 0) sm.flags[3] = (resident == 2) ? 1 : 0;
        team_reduce_vec<kVioPacked, NT - kErrTeam, T>(s.partials, s.nblocks, sm, tid);
        FLB_STAMP(1);
        if (!first && !resident) prior_commit(sm, pri, tid);
        if (multi) p2p_exchange<kVioPacked, T>(s.p2p, sm, p2p_tag, tid, s.timeout_flag);
        if (first && !resident) leader_prior<T>(sm, s.prior, tid);
        T::sync();
        if (tid < 32) {
            leader_fast_solve(sm, s.prm.sigma, -1.0, tid);                                // :871-878 (sign: :878)
            // The accepted outcome (*state += solution, :879) is formed while the error sum is still running, and -- in
            // the persistent kernel -- PUBLISHED right away: the accept test (:861) is the only thing the error sum
            // decides, everything else about the next pass (state, level, iteration) follows from the solve.  The
            // workers start the next pass on the accept branch; if the sum then says "reject" (at most once per
            // level: a rejection ends it) that pass is discarded and the corrected packet follows (see the kernel).
            // No speculation when the accept branch ends the update (nothing to overlap) or the solve failed.
            if (tid < 24) sm.xspec[tid] = reinterpret_cast<const double*>(&sm.x)[tid];
            __syncwarp();
            if (tid == 0) {
                state_boxplus(*reinterpret_cast<State18*>(sm.xspec), sm.sol);               // touches the 24 pose/bias doubles only
                const bool ok_p = sm.flags[3] == 0;
                const bool conv_p = !s.prm.force_all_passes && (norm3(sm.sol) * 57.3f < s.prm.conv_rot_deg) &&
                                    (norm3(sm.sol + 3) * 100.0f < s.prm.conv_pos_cm);
                const int it1 = c.iteration + 1;
                const bool done_p = conv_p || it1 >= s.prm.max_iteration;
                const bool stop_p = !ok_p || (done_p && (level - 1 < 0 || s.prm.single_level));
                const int spec = (pkt != nullptr && !stop_p) ? 1 : 0;
                sm.flags[4] = spec;
                sm.flags[5] = 0;
                if (spec) {
                    sm.cspec = c;
                    sm.cspec.level = done_p ? level - 1 : level;
                    sm.cspec.iteration = done_p ? 0 : it1;
                    sm.cspec.stop = 0;
                }
            }
            __syncwarp();
            const bool spec = sm.flags[4] != 0;
            if (spec) pkt_publish_warp<NC>(pkt, *reinterpret_cast<const State18*>(sm.xspec), &sm.cspec, flag, tid);
            FLB_STAMP(2);
            asm volatile("bar.sync 3, 64;" ::: "memory");                   // sm.error is ready
            FLB_STAMP(4);
            if (tid == 0) {
                const bool ok = sm.flags[3] == 0;
                // (the control block was initialised by k_vio_begin* / at kernel entry: level, last_error = total_residual, :755, :971)
                const long long nm = (long long)sm.packed[27];
                const float error = sm.error / (float)(unsigned long long)nm;              // :857
                c.passes[level] += 1;
                c.rows_total += nm;
                c.skipped_last = (int)sm.packed[28];
                bool EKF_end = false;
                int accept = 0;
                if (s.prm.force_all_passes || error <= c.last_error) {                     // :861
                    accept = 1;
                    c.last_error = error;
                    if (!s.prm.force_all_passes && (norm3(sm.sol) * 57.3f < s.prm.conv_rot_deg) &&
                        (norm3(sm.sol + 3) * 100.0f < s.prm.conv_pos_cm))
                        EKF_end = true;                                                    // :883
                    c.any_solved = 1;
                } else {
                    EKF_end = true;                                                        // :890
                }
                if (!ok) { EKF_end = true; c.status = -5; }
                c.iteration += 1;
                int docov = 0, newlevel = 0;
                if (EKF_end || c.iteration >= s.prm.max_iteration) {
                    // level finished -> ComputeJ advances (:974-977)
                    c.level_error[level] = c.last_error;
                    c.now_error = c.last_error;
                    c.level = level - 1;
                    c.iteration = 0;
                    c.last_error = 1e10f;
                    newlevel = 1;
                    if (s.prm.single_level) {
                        c.stop = 1;                                                         // UpdateState returns (:900)
                    } else if (c.level < 0 || !ok) {
                        c.stop = 1;
                        if (c.now_error < 1e10f && ok) { docov = 1; c.cov_updated = 1; }   // :978-981
                    }
                }
                c.err_buf = err_buf;
                sm.flags[0] = accept;
                sm.flags[1] = docov;
                sm.flags[2] = newlevel;
                if (spec && !accept) sm.flags[5] = 1;       // mispredicted: the pass now running is discarded
            }
            __syncwarp();
            FLB_STAMP(5);
            if (sm.flags[0]) {
                if (tid < 24) {
                    sm.xold[tid] = reinterpret_cast<const double*>(&sm.x)[tid];            // old_state = *state (:863)
                    reinterpret_cast<double*>(&sm.x)[tid] = sm.xspec[tid];                 // :879
                }
            } else {
                if (tid < 24) reinterpret_cast<double*>(&sm.x)[tid] = __ldcg(reinterpret_cast<const double*>(s.old_state) + tid);
            }                                                                              // *state = old_state (:890)
            __syncwarp();
            if (pkt && !spec) pkt_publish_warp<NC>(pkt, sm.x, &c, flag, tid);
            FLB_STAMP(6);
        }
    }
    __syncthreads();
}

// G_last holds HTH6 of the last ACCEPTED pass (the gain itself is only formed when :980 runs).
template <int NT>
__device__ __forceinline__ void vio_leader_finish(const VioSolveArgs& s, LeaderSmem& sm, const VioCtrl& c, bool first,
                                                  bool store_always, int resident) {
    const int tid = threadIdx.x;
    const int accept = sm.flags[0], docov = sm.flags[1], newlevel = sm.flags[2];
    if (accept) {
        if (tid < 24) reinterpret_cast<double*>(s.old_state)[tid] = sm.xold[tid];
        if (tid < 36) s.G_last[tid] = sm.packed[sym6_index(tid / 6, tid % 6)];
    }
    if (docov) {
        if (tid < 36) sm.HTH[tid] = accept ? sm.packed[sym6_index(tid / 6, tid % 6)] : __ldcg(s.G_last + tid);
        if (!first && !resident) load_cov_l2<NT>(&sm.x, s.state, tid);
        __syncthreads();
        leader_gain<Team<NT, false>>(sm, s.prm.sigma, tid);
        leader_cov_update(sm, sm.Gc, tid, NT);                                             // :980
    }
    if (c.stop || store_always) {
        store_state(s.state, &sm.x, tid, NT, docov != 0);
        if (tid == 0) *s.ctrl = c;
    }
    if (newlevel && tid < 24) reinterpret_cast<double*>(s.old_state)[tid] = reinterpret_cast<const double*>(&sm.x)[tid];   // :747 of the next level
}

__global__ void __launch_bounds__(32) k_vio_begin(VioCtrl* ctrl, int Pn_total) {
    if (threadIdx.x == 0) {
        VioCtrl c;
        c.level = 2;
        c.iteration = 0;
        c.stop = (Pn_total == 0) ? 1 : 0;                // :969-970
        c.last_error = 1e10f;
        c.now_error = 1e10f;
        c.any_solved = 0;
        for (int l = 0; l < 3; ++l) { c.passes[l] = 0; c.level_error[l] = 1e10f; }
        c.rows_total = 0;
        c.skipped_last = 0;
        c.cov_updated = 0;
        c.status = 0;
        c.err_buf = 0;
        *ctrl = c;
    }
}

__device__ __forceinline__ void vio_finalize_body(const VioSolveArgs& s) {
    __shared__ LeaderSmem sm;
    __shared__ VioCtrl c;
    __shared__ __align__(16) float s_err[kErrChunk];
    if (s.ctrl->stop) return;
    const int tid = threadIdx.x;
    if (tid == 0) c = *s.ctrl;
    load_poses_l2(&sm.x, s.state, &sm.xp, s.state_prop, tid);
    __syncthreads();
    const bool first = (c.passes[0] + c.passes[1] + c.passes[2]) == 0;
    vio_leader_solve<kLeaderBlock>(s, sm, c, s_err, first, nullptr, 0u, 0);
    vio_leader_finish<kLeaderBlock>(s, sm, c, first, true, 0);
}
__global__ void __launch_bounds__(kLeaderBlock) k_vio_finalize(VioSolveArgs s) { vio_finalize_body(s); }

// UpdateState(img, total_residual, level) alone: the control block starts at `level` with last_error = total_residual.
__global__ void __launch_bounds__(32) k_vio_begin_level(VioCtrl* ctrl, int Pn_total, int level, float total_residual) {
    if (threadIdx.x == 0) {
        VioCtrl c;
        c.level = level;
        c.iteration = 0;
        c.stop = (Pn_total == 0) ? 1 : 0;
        c.last_error = total_residual;
        c.now_error = total_residual;
        c.any_solved = 0;
        for (int l = 0; l < 3; ++l) { c.passes[l] = 0; c.level_error[l] = total_residual; }
        c.rows_total = 0;
        c.skipped_last = 0;
        c.cov_updated = 0;
        c.status = 0;
        c.err_buf = 0;
        *ctrl = c;
    }
}

// The member G of LidarSelector (:874): K_1[:, :6] * H_T_H[:6, :6] of the last ACCEPTED pass, formed from the stored
// H^T H block and the covariance the passes ran with.  out: 18 x 6 row-major (the other 12 columns of G are zero).
__global__ void __launch_bounds__(kLeaderBlock) k_vio_export_gain(VioSolveArgs s, double* out) {
    __shared__ LeaderSmem sm;
    const int tid = threadIdx.x;
    load_cov_l2<kLeaderBlock>(&sm.x, s.state, tid);
    if (tid == 0) sm.flags[3] = 0;
    if (tid < 36) sm.HTH[tid] = __ldcg(s.G_last + tid);
    __syncthreads();
    leader_prior<Team<kLeaderBlock, false>>(sm, s.prior, tid);
    __syncthreads();
    leader_gain<Team<kLeaderBlock, false>>(sm, s.prm.sigma, tid);
    for (int e = tid; e < kDim * 6; e += kLeaderBlock) out[e] = sm.Gc[e];
}
__global__ void __launch_bounds__(kLeaderBlock) k_vio_finalize_batched(const VioSolveArgs* __restrict__ args) {
    __shared__ VioSolveArgs s_s;
    {
        const unsigned* src = reinterpret_cast<const unsigned*>(args + blockIdx.x);
        unsigned* dst = reinterpret_cast<unsigned*>(&s_s);
        for (int e = threadIdx.x; e < (int)(sizeof(VioSolveArgs) / sizeof(unsigned)); e += kLeaderBlock) dst[e] = src[e];
    }
    __syncthreads();
    vio_finalize_body(s_s);
}
__global__ void k_vio_begin_batched(VioCtrl* const* ctrls, int B, int Pn_total) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    VioCtrl c;
    c.level = 2; c.iteration = 0; c.stop = (Pn_total == 0) ? 1 : 0;
    c.last_error = 1e10f; c.now_error = 1e10f; c.any_solved = 0;
    for (int l = 0; l < 3; ++l) { c.passes[l] = 0; c.level_error[l] = 1e10f; }
    c.rows_total = 0; c.skipped_last = 0; c.cov_updated = 0; c.status = 0; c.err_buf = 0;
    *ctrls[b] = c;
}

// =======================================================================================
// Persistent (one launch per update) kernels
// =======================================================================================
// All blocks are co-resident (cooperative launch, grid <= SMs x occupancy).  LIO / VIO: worker blocks + one
// dedicated leader block; a pass ends when every worker has arrived (red.release on a counter the leader
// acquire-polls), the leader runs the leader step above with its whole block and publishes the pose packet
// (below).  No host round trip, no empty launch.  Same pass and leader code as the kernel-per-pass path; the two
// group a pass's partial sums by different block sizes, so their states agree to rounding, not bit for bit.
// The IKFoM kernel still uses the classic form below (grid_arrive / grid_release / grid_wait: the last
// arriver becomes the leader and re-opens a generation barrier).
struct GridBarrier {
    unsigned int count;
    unsigned int gen;
    int timeout;
    int pad;
};

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(unsigned* p, unsigned v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Arrive; returns true (to every thread of the block) when this block is the last arriver.
__device__ __forceinline__ bool grid_arrive(GridBarrier* b, unsigned nblocks, unsigned* s_scratch /*2 words smem*/) {
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned g = ld_acquire_u32(&b->gen);
        __threadfence();
        const unsigned ticket = atomicAdd(&b->count, 1u);
        __threadfence();
        s_scratch[0] = (ticket == nblocks - 1) ? 1u : 0u;
        s_scratch[1] = g;
    }
    __syncthreads();
    return s_scratch[0] != 0;
}
// Leader: open the barrier.  Call with the whole block.
__device__ __forceinline__ void grid_release(GridBarrier* b, const unsigned* s_scratch) {
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        b->count = 0;
        __threadfence();
        st_release_u32(&b->gen, s_scratch[1] + 1u);
    }
    __syncthreads();
}
// Non-leader: wait.  A watchdog (~seconds) turns a would-be hang into FLB_ERR_TIMEOUT.
__device__ __forceinline__ bool grid_wait(GridBarrier* b, const unsigned* s_scratch) {
    __shared__ int s_ok;
    if (threadIdx.x == 0) {
        int ok = 1;
        unsigned long long spins = 0;
        while (ld_acquire_u32(&b->gen) == s_scratch[1]) {
            __nanosleep(20);
            if (++spins > 3000000ull) { ok = 0; b->timeout = 1; break; }
            if ((spins & 0xffff) == 0 && *((volatile int*)&b->timeout)) { ok = 0; break; }
        }
        s_ok = ok;
    }
    __syncthreads();
    return s_ok != 0;
}

// ---------------------------------------------------------------------------------------
// Pose packet: barrier release and state broadcast in one L2 round trip
// ---------------------------------------------------------------------------------------
// The leader does not "open" a barrier and let every block re-read state and control from global
// memory (three dependent L2 round trips per pass).  It publishes the new 24 pose/bias doubles and
// the control block as 8-byte units {payload word, flag} with flag = epoch + pass number; a waiting
// block polls the units themselves, so the first successful poll already carries the data (the
// 8-byte unit is written and read by single instructions, so payload and flag travel together).
// The leader is always the same block, so whatever it needs from pass to pass (prior block, covariance, VIO
// old_state / G_last, exchange counter) stays in its shared memory or is re-read by the block that wrote it.
// The arrive counter runs up monotonically during a launch (the leader waits for nworkers * (pass + 1)) and
// is zeroed by the leader on the stopping pass.
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
// Waiting block: warp 0 polls, then the words go to x / c in shared memory.  Returns false (to the
// whole block) when the watchdog (~seconds) tripped: a would-be hang becomes FLB_ERR_TIMEOUT.
template <int NC>
__device__ __forceinline__ bool pkt_wait(const unsigned long long* pkt, State18& x, void* c, unsigned flag, GridBarrier* b,
                                         unsigned* s_scratch, unsigned long long spin_limit = 3000000ull) {
    constexpr int N = kStateWords + NC;
    constexpr int PER = (N + 31) / 32;
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        unsigned long long v[PER];
        unsigned long long spins = 0;
        bool good = true;
        for (;;) {
            bool ok = true;
#pragma unroll
            for (int u = 0; u < PER; ++u) {
                const int e = lane + 32 * u;
                if (e < N) {
                    v[u] = ld_relaxed_u64(pkt + e);
                    ok = ok && ((unsigned)(v[u] >> 32) == flag);
                }
            }
            if (__all_sync(0xffffffffu, ok)) break;
            __nanosleep(20);
            ++spins;
            bool bail = false;
            if (spins > spin_limit) { b->timeout = 1; bail = true; }
            else if ((spins & 0xffff) == 0 && *((volatile int*)&b->timeout)) bail = true;
            if (__any_sync(0xffffffffu, bail)) { good = false; break; }
        }
        if (good) {
            unsigned* xs = reinterpret_cast<unsigned*>(&x);
            unsigned* cs = reinterpret_cast<unsigned*>(c);
#pragma unroll
            for (int u = 0; u < PER; ++u) {
                const int e = lane + 32 * u;
                if (e < N) {
                    if (e < kStateWords) xs[e] = (unsigned)v[u];
                    else cs[e - kStateWords] = (unsigned)v[u];
                }
            }
        }
        if (lane == 0) s_scratch[1] = good ? 1u : 0u;
    }
    __syncthreads();
    return s_scratch[1] != 0;
}

__device__ __forceinline__ void lio_pose_from(const LioParamsDev& prm, const State18& x, LioPose& pose) {
    for (int i = 0; i < 9; ++i) { pose.R[i] = x.rot[i]; pose.R_LI[i] = prm.R_LI[i]; }
    for (int i = 0; i < 3; ++i) { pose.p[i] = x.pos[i]; pose.t_LI[i] = prm.t_LI[i]; }
    m3_T(pose.R, pose.Rt);
    m3_T(pose.R_LI, pose.RLIt);
}

// Leader block of a persistent kernel, before the first pass has even arrived: fetch the covariance and form
// the prior block (P11^-1, P21 P11^-1) in shared memory, where both stay for the whole update.
// Returns 1, or 2 when the prior is singular.
template <int NT>
__device__ __forceinline__ int leader_prepare(LeaderSmem& sm, const State18* state, PriorBlock* prior_g) {
    const int tid = threadIdx.x;
    load_cov_l2<NT>(&sm.x, state, tid);
    if (tid == 0) sm.flags[3] = 0;
    __syncthreads();
    leader_prior<Team<NT, false>>(sm, prior_g, tid);
    __syncthreads();
    return sm.flags[3] ? 2 : 1;
}

// Workers: arrive (release) without waiting for the ticket.
__device__ __forceinline__ void grid_arrive_release(GridBarrier* b) {
    __syncthreads();
    if (threadIdx.x == 0) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(&b->count) : "memory");
}
// Leader block: wait until `target` arrivals have been counted (acquire).  False when the watchdog tripped.
__device__ __forceinline__ bool leader_wait_arrivals(GridBarrier* b, unsigned target, unsigned* s_scratch) {
    if (threadIdx.x == 0) {
        unsigned ok = 1u;
        unsigned long long spins = 0;
        while (ld_acquire_u32(&b->count) != target) {
            if (++spins > 40000000ull) { ok = 0u; b->timeout = 1; break; }
            if ((spins & 0xffff) == 0 && *((volatile int*)&b->timeout)) { ok = 0u; break; }
        }
        s_scratch[1] = ok;
    }
    __syncthreads();
    return s_scratch[1] != 0u;
}

// ---------------------------------------------------------------------------------------
// LIO: whole iterated update in one launch
// ---------------------------------------------------------------------------------------
// Grid = worker blocks + ONE leader block (the last one).  The leader owns no points: it waits for the
// arrivals of each pass, reduces, solves and publishes the pose packet.  Keeping the leader on one SM
// keeps its code and its constants (prior block, state_propagat, covariance) warm from pass to pass;
// a last-arriver leader would run the solve on a different, cold SM every pass.
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK, 1) k_lio_update_persistent(LioArgs a, LioSolveArgs s, GridBarrier* bar,
                                                                 unsigned long long* pkt, unsigned epoch,
                                                                 unsigned long long* trace, unsigned long long* dbg) {
    constexpr int K = lio_packed(6);
    constexpr int NC = (int)(sizeof(LioCtrl) / sizeof(unsigned));
    __shared__ LioPose s_pose;
    __shared__ double s_acc[BLOCK / 32][K];
    __shared__ unsigned s_bar[2];
    __shared__ LeaderSmem sm;
    __shared__ LioCtrl s_ctrl;       // block-local mirror of the loop state (src/laserMapping.cpp:1472-1473, :1506)
    __shared__ int s_rows[18][BLOCK];
    __shared__ unsigned long long s_seq_base;
    const int tid = threadIdx.x;
    const int nworkers = (int)gridDim.x - 1;
    const bool is_leader = (int)blockIdx.x == nworkers;
    const bool multi = s.p2p.world > 1;
    bool first = true;
    int pass_no = 0;
    if (trace && blockIdx.x == 0 && tid == 0) trace[0] = global_ns();
    if (tid == 96) s_seq_base = multi ? *s.p2p.seq : 0ull;     // exchange counter: identical on every rank
    // every block keeps the pose/bias part of state and state_propagat resident in shared memory
    const State18* x_src = s.init_x ? s.init_x : s.state;
    const State18* xp_src = s.init_xp ? s.init_xp : s.state_prop;
    if (tid < 24) reinterpret_cast<double*>(&sm.x)[tid] = reinterpret_cast<const double*>(x_src)[tid];
    else if (tid < 48) reinterpret_cast<double*>(&sm.xp)[tid - 24] = reinterpret_cast<const double*>(xp_src)[tid - 24];
    if (tid == 64) {
        LioCtrl c;
        c.iterCount = -1; c.rematch_num = 0; c.nearest_search_en = 1; c.stop = 0;
        c.passes = c.knn_passes = c.n_eff_last = c.converged_last = 0; c.status = 0;
        c.res_mean_last = 0.0; c.rows_total = 0;
        s_ctrl = c;
    }
    __syncthreads();
    int resident = 0;
    if (is_leader) {
        warm_pages(a.warm, tid, BLOCK);
        if (s.init_x) {                  // the pending reset: state / state_prop take the saved pair (whole structs)
            const double* a0 = reinterpret_cast<const double*>(s.init_x);
            const double* a1 = reinterpret_cast<const double*>(s.init_xp);
            double* d0 = reinterpret_cast<double*>(s.state);
            double* d1 = reinterpret_cast<double*>(const_cast<State18*>(s.state_prop));
            for (int e = tid; e < (int)(sizeof(State18) / sizeof(double)); e += BLOCK) { d0[e] = a0[e]; d1[e] = a1[e]; }
        }
        resident = leader_prepare<BLOCK>(sm, x_src, s.prior);
    } else if (a.prefetch) {
        // A map larger than a few MB is cold in L2 when the frame starts (other work ran in between): the kNN walk
        // would then pay one DRAM latency per dependent step.  Stream the sorted points and the cell table into L2
        // with bulk prefetches (asynchronous: nobody waits for them), 4 KB per instruction.
        const size_t nb_pts = (size_t)a.M * sizeof(float4);
        const size_t nb_cells = ((size_t)a.grid.nx * a.grid.ny * a.grid.nz + 1) * sizeof(int) / 16 * 16;
        const size_t step = 4096, stride = (size_t)nworkers * BLOCK * step;
        for (size_t off = ((size_t)blockIdx.x * BLOCK + tid) * step; off < nb_pts; off += stride)
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<const char*>(a.map_pts) + off),
                         "r"((unsigned)min(step, nb_pts - off)) : "memory");
        for (size_t off = ((size_t)blockIdx.x * BLOCK + tid) * step; off < nb_cells; off += stride)
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<const char*>(a.cell_start) + off),
                         "r"((unsigned)min(step, nb_cells - off)) : "memory");
    }
    for (;;) {
        const unsigned flag = epoch + (unsigned)pass_no + 1u;
        if (is_leader) {
            if (!leader_wait_arrivals(bar, (unsigned)nworkers * (unsigned)(pass_no + 1), s_bar)) return;
            if (trace && tid == 0 && 2 + 2 * pass_no < kTraceLen) trace[1 + 2 * pass_no] = global_ns();
            unsigned long long* fine = (trace && 64 + 8 * pass_no + 8 <= kTraceLen) ? trace + 64 + 8 * pass_no : nullptr;
            const unsigned p2p_tag = multi ? ((unsigned)(s_seq_base + (unsigned long long)pass_no + 1ull) | 0x80000000u) : 0u;
            lio_leader_solve<BLOCK>(s, sm, s_ctrl, first, pkt, flag, resident, fine, p2p_tag);
            if (trace && tid == 0 && 2 + 2 * pass_no < kTraceLen) trace[2 + 2 * pass_no] = global_ns();
            lio_leader_finish<BLOCK>(s, sm, s_ctrl, first, false, resident, fine);
            if (s_ctrl.stop && tid == 0) {
                bar->count = 0;
                if (multi) *s.p2p.seq = s_seq_base + (unsigned long long)pass_no + 1ull;
            }
        } else {
            if (dbg && tid == 0) dbg[blockIdx.x * 16 + 0] = global_ns();
            if (tid == 0) lio_pose_from(a.prm, sm.x, s_pose);
            __syncthreads();
            if (dbg && tid == 0) dbg[blockIdx.x * 16 + 1] = global_ns();
            const int nearest = s_ctrl.nearest_search_en;
            double acc[K];
#pragma unroll
            for (int k = 0; k < K; ++k) acc[k] = 0.0;
            // Morton-contiguous chunks of a.chunk <= 32 points (sized by the host so that every warp of every
            // worker gets one chunk when N allows: the pass is latency-bound, so spreading the points over all
            // warps beats filling lanes) dealt round-robin to the worker blocks; the chunk -> thread map is the
            // same in every pass, so each thread re-reads only its own per-point cache entries.
            for (int c = (tid >> 5) * nworkers + blockIdx.x; c * a.chunk < a.N; c += (BLOCK / 32) * nworkers) {
                const int i = c * a.chunk + (tid & 31);
                if ((tid & 31) < a.chunk && i < a.N) {
                    bool active;
                    double row[6], z, absres;
                    lio_point<6>(a, s_pose, nearest != 0, i, active, row, z, absres, &s_rows[0][tid], BLOCK);
                    if (active) lio_accumulate<6>(acc, row, z, absres);
                }
            }
            if (dbg && (tid & 31) == 0) dbg[blockIdx.x * 16 + 4 + (tid >> 5)] = global_ns();   // per warp: compute done
            block_reduce_store<K, BLOCK>(acc, s_acc, a.partials);
            if (dbg && tid == 0) dbg[blockIdx.x * 16 + 2] = global_ns();
            grid_arrive_release(bar);
            if (dbg && tid == 0) dbg[blockIdx.x * 16 + 3] = global_ns();
            if (!pkt_wait<NC>(pkt, sm.x, &s_ctrl, flag, bar, s_bar, multi ? 40000000ull : 3000000ull)) return;
        }
        first = false;
        ++pass_no;
        if (s_ctrl.stop) break;
    }
}

// ---------------------------------------------------------------------------------------
// VIO: ComputeJ (3 levels x up to T passes) in one launch  (same worker / leader split)
// ---------------------------------------------------------------------------------------
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK, 1) k_vio_update_persistent(VioArgs a, VioSolveArgs s, GridBarrier* bar,
                                                                    unsigned long long* pkt, unsigned epoch,
                                                                    unsigned long long* trace, unsigned long long* dbg, int err_cap) {
    constexpr int NW = BLOCK / 32;
    constexpr int NC = (int)(sizeof(VioCtrl) / sizeof(unsigned));
    __shared__ VioPose s_pose;
    __shared__ float s_lat[NW][128];
    __shared__ double s_res[NW][64];
    __shared__ double s_acc[NW][kVioPacked];
    __shared__ unsigned s_bar[2];
    __shared__ LeaderSmem sm;
    __shared__ VioCtrl s_ctrl;
    extern __shared__ __align__(128) float s_err[];    // dynamic: the LEADER's staging of the per-patch errors (err_cap floats)
    __shared__ unsigned long long s_seq_base;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int nworkers = (int)gridDim.x - 1;
    const bool is_leader = (int)blockIdx.x == nworkers;
    const int Pn = a.Pn_dev ? min(*a.Pn_dev, a.Pn) : a.Pn;     // device-built patch list: its length lives on the device
    if (Pn <= 0 && s.p2p.world <= 1) {                         // :969-970 (the host short-circuits when it knows)
        if (is_leader && s.prior_from_state) {
            const double* a0 = reinterpret_cast<const double*>(s.state);
            double* d1 = reinterpret_cast<double*>(const_cast<State18*>(s.state_prop));
            for (int e = tid; e < (int)(sizeof(State18) / sizeof(double)); e += BLOCK) d1[e] = a0[e];
        }
        if (is_leader && tid == 0) {
            VioCtrl c;
            c.level = 2; c.iteration = 0; c.stop = 1;
            c.last_error = 1e10f; c.now_error = 1e10f; c.any_solved = 0;
            for (int l = 0; l < 3; ++l) { c.passes[l] = 0; c.level_error[l] = 1e10f; }
            c.rows_total = 0; c.skipped_last = 0; c.cov_updated = 0; c.status = 0; c.err_buf = 0;
            *s.ctrl = c;
        }
        return;
    }
    const bool multi = s.p2p.world > 1;
    bool first = true;
    int pass_no = 0;
    if (trace && blockIdx.x == 0 && tid == 0) trace[0] = global_ns();
    if (tid == 96) s_seq_base = multi ? *s.p2p.seq : 0ull;     // exchange counter: identical on every rank
    const State18* xp_src = s.prior_from_state ? s.state : s.state_prop;
    if (tid < 24) reinterpret_cast<double*>(&sm.x)[tid] = reinterpret_cast<const double*>(s.state)[tid];
    else if (tid < 48) reinterpret_cast<double*>(&sm.xp)[tid - 24] = reinterpret_cast<const double*>(xp_src)[tid - 24];
    if (tid == 64) {
        VioCtrl c;
        c.level = 2; c.iteration = 0; c.stop = 0;
        c.last_error = 1e10f; c.now_error = 1e10f; c.any_solved = 0;
        for (int l = 0; l < 3; ++l) { c.passes[l] = 0; c.level_error[l] = 1e10f; }
        c.rows_total = 0; c.skipped_last = 0; c.cov_updated = 0; c.status = 0; c.err_buf = 0;
        s_ctrl = c;
    }
    // every warp owns at most one patch: its pose-independent inputs stay in registers for all passes
    const bool single = nworkers * NW >= Pn;
    PatchIn pin;
    if (single && !is_leader && blockIdx.x * NW + warp < Pn) vio_patch_load(a, blockIdx.x * NW + warp, tid & 31, pin);
    __syncthreads();
    int resident = 0;
    if (is_leader) {
        warm_pages(a.warm, tid, BLOCK);
        if (s.prior_from_state) {        // the pending `state_propagat = state`: the whole struct, before anything writes *state
            const double* a0 = reinterpret_cast<const double*>(s.state);
            double* d1 = reinterpret_cast<double*>(const_cast<State18*>(s.state_prop));
            for (int e = tid; e < (int)(sizeof(State18) / sizeof(double)); e += BLOCK) d1[e] = a0[e];
        }
        resident = leader_prepare<BLOCK>(sm, s.state, s.prior);
    }
    for (;;) {
        const unsigned flag = epoch + (unsigned)pass_no + 1u;
        const unsigned p2p_tag = multi ? ((unsigned)(s_seq_base + (unsigned long long)pass_no + 1ull) | 0x80000000u) : 0u;
        if (is_leader) {
            if (!leader_wait_arrivals(bar, (unsigned)nworkers * (unsigned)(pass_no + 1), s_bar)) return;
            if (trace && tid == 0 && 2 + 2 * pass_no < kTraceLen) trace[1 + 2 * pass_no] = global_ns();
            unsigned long long* fine = (trace && 32 + 8 * pass_no + 8 <= kTraceLen) ? trace + 32 + 8 * pass_no : nullptr;
            vio_leader_solve<BLOCK>(s, sm, s_ctrl, s_err, first, pkt, flag, resident, fine, p2p_tag, pass_no & 1, err_cap, Pn);
            if (trace && tid == 0 && 2 + 2 * pass_no < kTraceLen) trace[2 + 2 * pass_no] = global_ns();
            vio_leader_finish<BLOCK>(s, sm, s_ctrl, first, false, resident);
            if (sm.flags[5]) {
                // The error sum rejected the step whose accept branch was published ahead of it (:861 / :890): the
                // pass now running started from the wrong state.  Wait for it, drop it, publish the real
                // continuation (the rejected step's old_state at the next level, or stop).  Fused multi-GPU mode:
                // every rank mispredicts identically; one (payload-free) exchange keeps the mailbox parity rule.
                ++pass_no;
                if (!leader_wait_arrivals(bar, (unsigned)nworkers * (unsigned)(pass_no + 1), s_bar)) return;
                if (trace && tid == 0 && 2 + 2 * pass_no < kTraceLen) trace[1 + 2 * pass_no] = global_ns();
                if (multi) {
                    const unsigned tag2 = (unsigned)(s_seq_base + (unsigned long long)pass_no + 1ull) | 0x80000000u;
                    p2p_exchange<kVioPacked, Team<BLOCK, false>>(s.p2p, sm, tag2, tid, s.timeout_flag);
                }
                if (tid < 32) pkt_publish_warp<NC>(pkt, sm.x, &s_ctrl, epoch + (unsigned)pass_no + 1u, tid);
                if (trace && tid == 0 && 2 + 2 * pass_no < kTraceLen) trace[2 + 2 * pass_no] = global_ns();
                __syncthreads();
            }
            if (s_ctrl.stop && tid == 0) {
                bar->count = 0;
                if (multi) *s.p2p.seq = s_seq_base + (unsigned long long)pass_no + 1ull;
            }
        } else {
            if (dbg && tid == 0) dbg[blockIdx.x * kVioDbg + 0] = global_ns();
            // fused multi-GPU mode: this rank's patch count of the pass goes out first (the leaders size their gather by it)
            if (multi && blockIdx.x == 0 && tid >= 32 && tid < 32 + s.p2p.world)
                ll_store_line(&s.p2p.mail[tid - 32]->sums[p2p_tag & 1u][s.p2p.rank][31], (double)Pn, p2p_tag);
            if (tid == 0) vio_make_pose(a.prm.Rci, a.prm.Pci, a.prm.Jdphi_dR, a.prm.Jdp_dR, sm.x.rot, sm.x.pos, s_pose);
            __syncthreads();
            if (dbg && tid == 0) dbg[blockIdx.x * kVioDbg + 1] = global_ns();
            const int level = s_ctrl.level;
            double accv = 0.0, n_meas = 0.0, skipped = 0.0;
            // the leader reads the per-patch errors as self-validating units, so the error chain of a warp's LAST patch of
            // the pass can run after the block has arrived (it only feeds the error sum, which is off the critical path)
            const unsigned utag = (!multi && a.err_units) ? (flag | 0x80000000u) : 0u;
            const bool can_defer = multi || utag != 0u;
            int pend_i = -1;
            bool pend_tiny = false;
            unsigned long long* wd = dbg ? dbg + blockIdx.x * kVioDbg + 8 + 4 * warp : nullptr;
            for (int i = blockIdx.x * NW + warp; i < Pn; i += nworkers * NW) {
                if (!single) vio_patch_load(a, i, tid & 31, pin);
                const bool last = can_defer && (i + nworkers * NW >= Pn);
                if (vio_patch(a, s_pose, level, i, pin, s_lat[warp], s_res[warp], accv, n_meas, skipped, wd, p2p_tag, pass_no & 1, utag, last,
                              &pend_tiny))
                    pend_i = i;
            }
            vio_block_reduce_store<BLOCK>(accv, n_meas, skipped, s_acc, a.partials);
            if (dbg && tid == 0) dbg[blockIdx.x * kVioDbg + 2] = global_ns();
            grid_arrive_release(bar);
            if (dbg && tid == 0) dbg[blockIdx.x * kVioDbg + 3] = global_ns();
            if (pend_i >= 0) vio_patch_error(a, pend_i, s_res[warp], pend_tiny, p2p_tag, utag, pass_no & 1, wd);
            if (!pkt_wait<NC>(pkt, sm.x, &s_ctrl, flag, bar, s_bar, multi ? 40000000ull : 3000000ull)) return;
        }
        first = false;
        ++pass_no;
        if (s_ctrl.stop) break;
    }
}

// =======================================================================================
// IMU forward propagation + backward undistortion (SURVEY.md section 8 row f3):
// ImuProcess::UndistortPcl from src/IMU_Processing.cpp:655 on.
// =======================================================================================
struct ImuSampleDev { double t, gyr[3], acc[3]; };            // == flb_imu_sample
struct ImuCarryDev { double last_lidar_end_time, acc_s_last[3], angvel_last[3]; };   // == flb_imu_carry
struct ImuAux { double extR_Ri[9], exrR_extT[3], pos_end[3]; int n_poses; int pad; };

// One block.  The loop over IMU samples is sequential by nature (K ~ 10-50 per frame); thread 0 carries the
// 3-vectors and builds F_x / cov_w, all threads do the two 18x18x18 products of
// cov = F cov F^T + cov_w (:720), summed in the reference's (Eigen's) index order.
__global__ void __launch_bounds__(352) k_imu_propagate(State18* x, const ImuSampleDev* v_imu, int n_imu, ImuParamsDev prm,
                                                       double pcl_beg_time, double pcl_end_time, ImuCarryDev* carry,
                                                       ImuPose* poses, ImuAux* aux) {
    __shared__ double P[324], T[324], F[324], W[324];
    __shared__ double R_imu[9], vel_imu[3], pos_imu[3], acc_imu[3], angvel_avr[3];
    __shared__ int s_skip, s_np;
    const int tid = threadIdx.x;
    if (tid < 324) P[tid] = x->cov[tid];
    if (tid == 0) {
        for (int k = 0; k < 9; ++k) R_imu[k] = x->rot[k];
        for (int k = 0; k < 3; ++k) {
            vel_imu[k] = x->vel[k]; pos_imu[k] = x->pos[k];
            acc_imu[k] = carry->acc_s_last[k]; angvel_avr[k] = carry->angvel_last[k];
        }
        ImuPose p0;                                                               // :658
        p0.t = 0.0;
        for (int k = 0; k < 3; ++k) { p0.acc[k] = acc_imu[k]; p0.gyr[k] = angvel_avr[k]; p0.vel[k] = vel_imu[k]; p0.pos[k] = pos_imu[k]; }
        for (int k = 0; k < 9; ++k) p0.rot[k] = R_imu[k];
        poses[0] = p0;
        s_np = 1;
    }
    __syncthreads();
    const double last_end = carry->last_lidar_end_time;
    for (int it = 0; it + 1 < n_imu; ++it) {                                      // :666
        if (tid < 324) { F[tid] = ((tid / 18) == (tid % 18)) ? 1.0 : 0.0; W[tid] = 0.0; }
        __syncthreads();
        if (tid == 0) {
            const ImuSampleDev head = v_imu[it], tail = v_imu[it + 1];
            s_skip = (tail.t < last_end) ? 1 : 0;                                 // :671
            if (!s_skip) {
                double acc_avr[3];
                for (int k = 0; k < 3; ++k) {
                    angvel_avr[k] = 0.5 * (head.gyr[k] + tail.gyr[k]);            // :673-681
                    acc_avr[k] = 0.5 * (head.acc[k] + tail.acc[k]);
                }
                for (int k = 0; k < 3; ++k) {
                    angvel_avr[k] -= x->bg[k];                                    // :687
                    acc_avr[k] = acc_avr[k] * prm.G_m_s2 / prm.mean_acc_norm - x->ba[k];   // :688
                }
                const double dt = (head.t < last_end) ? (tail.t - last_end) : (tail.t - head.t);   // :690-697
                double Exp_f[9], Exp_m[9], askew[9], Ra[9];
                so3_exp_dt(angvel_avr, dt, Exp_f);                                // :701
                so3_exp_dt(angvel_avr, -dt, Exp_m);                               // :707
                skew3(acc_avr, askew);
                m3_mul(R_imu, askew, Ra);
                for (int i = 0; i < 3; ++i)
                    for (int j = 0; j < 3; ++j) {
                        F[i * 18 + j] = Exp_m[i * 3 + j];                         // (0,0)
                        F[i * 18 + 9 + j] = (i == j) ? -dt : 0.0;                 // (0,9)  = -I dt
                        F[(3 + i) * 18 + 6 + j] = (i == j) ? dt : 0.0;            // (3,6)  =  I dt
                        F[(6 + i) * 18 + j] = -Ra[i * 3 + j] * dt;                // (6,0)  = -R [a]x dt
                        F[(6 + i) * 18 + 12 + j] = -R_imu[i * 3 + j] * dt;        // (6,12) = -R dt
                        F[(6 + i) * 18 + 15 + j] = (i == j) ? dt : 0.0;           // (6,15) =  I dt
                    }
                for (int i = 0; i < 3; ++i) {
                    W[i * 18 + i] = prm.cov_gyr[i] * dt * dt;                     // :715
                    W[(9 + i) * 18 + 9 + i] = prm.cov_bias_gyr[i] * dt * dt;      // :717
                    W[(12 + i) * 18 + 12 + i] = prm.cov_bias_acc[i] * dt * dt;    // :718
                }
                {
                    double RD[9], Rt[9], RDRt[9];                                 // :716, left to right
                    for (int i = 0; i < 3; ++i)
                        for (int j = 0; j < 3; ++j) RD[i * 3 + j] = R_imu[i * 3 + j] * prm.cov_acc[j];
                    m3_T(R_imu, Rt);
                    m3_mul(RD, Rt, RDRt);
                    for (int i = 0; i < 3; ++i)
                        for (int j = 0; j < 3; ++j) W[(6 + i) * 18 + 6 + j] = RDRt[i * 3 + j] * dt * dt;
                }
                double Rn[9], Ra_v[3];
                m3_mul(R_imu, Exp_f, Rn);                                         // :723
                for (int k = 0; k < 9; ++k) R_imu[k] = Rn[k];
                m3_vec(R_imu, acc_avr, Ra_v);
                for (int k = 0; k < 3; ++k) acc_imu[k] = Ra_v[k] + x->grav[k];    // :726
                for (int k = 0; k < 3; ++k) pos_imu[k] = pos_imu[k] + vel_imu[k] * dt + 0.5 * acc_imu[k] * dt * dt;   // :729
                for (int k = 0; k < 3; ++k) vel_imu[k] = vel_imu[k] + acc_imu[k] * dt;   // :732
                ImuPose p;
                p.t = tail.t - pcl_beg_time;                                      // :737
                for (int k = 0; k < 3; ++k) { p.acc[k] = acc_imu[k]; p.gyr[k] = angvel_avr[k]; p.vel[k] = vel_imu[k]; p.pos[k] = pos_imu[k]; }
                for (int k = 0; k < 9; ++k) p.rot[k] = R_imu[k];
                poses[s_np] = p;
                s_np = s_np + 1;
            }
        }
        __syncthreads();
        if (s_skip) continue;
        if (tid < 324) {                                                          // cov = F cov F^T + cov_w, :720
            const int i = tid / 18, j = tid % 18;
            double acc = 0.0;
            for (int k = 0; k < 18; ++k) acc += F[i * 18 + k] * P[k * 18 + j];
            T[tid] = acc;
        }
        __syncthreads();
        if (tid < 324) {
            const int i = tid / 18, j = tid % 18;
            double acc = 0.0;
            for (int k = 0; k < 18; ++k) acc += T[i * 18 + k] * F[j * 18 + k];
            P[tid] = acc + W[tid];
        }
        __syncthreads();
    }
    if (tid < 324) x->cov[tid] = P[tid];
    if (tid == 0) {
        // frame-end prediction, :743-758
        const double imu_end_time = v_imu[n_imu - 1].t;
        double note, dt;
        if (imu_end_time > pcl_beg_time) {
            note = pcl_end_time > imu_end_time ? 1.0 : -1.0;
            dt = note * (pcl_end_time - imu_end_time);
        } else {
            note = pcl_end_time > pcl_beg_time ? 1.0 : -1.0;
            dt = note * (pcl_end_time - pcl_beg_time);
        }
        const double w[3] = {note * angvel_avr[0], note * angvel_avr[1], note * angvel_avr[2]};
        double E[9], Rn[9];
        so3_exp_dt(w, dt, E);
        m3_mul(R_imu, E, Rn);
        for (int k = 0; k < 3; ++k) {
            x->vel[k] = vel_imu[k] + note * acc_imu[k] * dt;
            x->pos[k] = pos_imu[k] + note * vel_imu[k] * dt + note * 0.5 * acc_imu[k] * dt * dt;
        }
        for (int k = 0; k < 9; ++k) x->rot[k] = Rn[k];
        for (int k = 0; k < 3; ++k) { carry->acc_s_last[k] = acc_imu[k]; carry->angvel_last[k] = angvel_avr[k]; }   // :735-736
        carry->last_lidar_end_time = pcl_end_time;                                // :761
        double RLIt[9], rot_end_T[9];
        m3_T(prm.R_LI, RLIt);
        m3_T(Rn, rot_end_T);
        m3_mul(RLIt, rot_end_T, aux->extR_Ri);                                    // :763
        m3_vec(RLIt, prm.t_LI, aux->exrR_extT);                                   // :764
        for (int k = 0; k < 3; ++k) aux->pos_end[k] = x->pos[k];
        aux->n_poses = s_np;
    }
}

// Backward pass, :778-808.  The reference walks the time-ordered points from the last one down with a pose
// cursor that only moves to earlier IMU poses: point i is compensated with head H_i = min over j >= i of
// v_j, v_j = the last pose whose offset_time is < t_j (-1: none, the walk has ended and the remaining points
// stay as they are).  v is per point, the suffix minimum is one scan, the compensation is per point again.
__global__ void k_imu_heads(const float* __restrict__ offset_ms, int os, int n, const ImuPose* __restrict__ poses,
                            const ImuAux* __restrict__ aux, int* __restrict__ heads) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double t = (double)offset_ms[(size_t)i * os] / double(1000);
    int v = -1;
    for (int H = aux->n_poses - 2; H >= 0; --H)
        if (t > poses[H].t) { v = H; break; }
    heads[i] = v;
}

// In-place suffix minimum of heads[0..n) by one block.
__global__ void __launch_bounds__(1024) k_suffix_min(int* __restrict__ heads, int n) {
    __shared__ int smin[1024];
    const int tid = threadIdx.x;
    const int per = (n + 1023) / 1024;
    const int a = min(n, tid * per), b = min(n, a + per);
    int m = 0x7fffffff;
    for (int i = a; i < b; ++i) m = min(m, heads[i]);
    smin[tid] = m;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {            // inclusive suffix scan of the segment minima
        const int o = (tid + off < 1024) ? smin[tid + off] : 0x7fffffff;
        __syncthreads();
        smin[tid] = min(smin[tid], o);
        __syncthreads();
    }
    int run = (tid + 1 < 1024) ? smin[tid + 1] : 0x7fffffff;
    for (int i = b - 1; i >= a; --i) {
        run = min(run, heads[i]);
        heads[i] = run;
    }
}

__global__ void k_imu_undistort(const float* __restrict__ in_xyz, int stride, const float* __restrict__ offset_ms, int os, int n,
                                const ImuPose* __restrict__ poses, const ImuAux* __restrict__ aux, const int* __restrict__ heads,
                                ImuParamsDev prm, float4* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float p[3] = {in_xyz[(size_t)i * stride], in_xyz[(size_t)i * stride + 1], in_xyz[(size_t)i * stride + 2]};
    const float off = offset_ms[(size_t)i * os];
    const double t = (double)off / double(1000);
    const int H = heads[i];
    if (H >= 0) {
        imu_compensate_point(poses[H], prm.R_LI, prm.t_LI, aux->extR_Ri, aux->exrR_extT, aux->pos_end, t, p);
        // The first point is the reference's loop exit (:807): the outer loop still visits the earlier poses and
        // compensates that point again for every one of them that precedes it in time.
        if (i == 0)
            for (int h = H - 1; h >= 0; --h)
                if (t > poses[h].t) imu_compensate_point(poses[h], prm.R_LI, prm.t_LI, aux->extR_Ri, aux->exrR_extT, aux->pos_end, t, p);
    }
    out[i] = make_float4(p[0], p[1], p[2], off);
}

// =======================================================================================
// Visual-map growth, candidate scoring (SURVEY.md section 8 row f4): first loop of
// LidarSelector::addSparseMap, src/lidar_selection.cpp:150-168.
// =======================================================================================
// The reference walks the points in order and lets a point take its grid cell when its score is strictly above
// the cell's current value.  The outcome per cell is "the first point that reaches the cell's maximum, if that
// maximum exceeds the incoming value": one 64-bit atomicMax per point on {order-preserving score bits,
// ~index}; the seed carries index bits 0xFFFFFFFF so that an equal score never displaces it (a candidate's index bits
// are 0xFFFFFFFE - i: point 0 must stay distinguishable from the seed).
__device__ __forceinline__ unsigned ordered_f32(float f) {
    const unsigned b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float unordered_f32(unsigned o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o);
}
__global__ void k_vmap_seed(const float* __restrict__ map_value, int ncell, unsigned long long* __restrict__ key) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < ncell) key[c] = ((unsigned long long)ordered_f32(map_value[c]) << 32) | 0xFFFFFFFFull;
}
__global__ void k_vmap_candidates(CamModel cam, const double* __restrict__ Rcw_Pcw, const unsigned char* __restrict__ img,
                                  const float* __restrict__ xyz, int n, int grid_size, int grid_n_height, int border,
                                  unsigned long long* __restrict__ key) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double Rcw[9], Pcw[3];
#pragma unroll
    for (int k = 0; k < 9; ++k) Rcw[k] = Rcw_Pcw[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) Pcw[k] = Rcw_Pcw[9 + k];
    float score = 0.0f;
    const float p[3] = {xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2]};
    const int cell = visual_candidate(cam, Rcw, Pcw, img, cam.width, p, grid_size, grid_n_height, border, &score);
    if (cell < 0) return;
    atomicMax(key + cell, ((unsigned long long)ordered_f32(score) << 32) | (unsigned long long)(0xFFFFFFFEu - (unsigned)i));
}
__global__ void k_vmap_resolve(const unsigned long long* __restrict__ key, int ncell, float* __restrict__ map_value,
                               int* __restrict__ winner) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncell) return;
    const unsigned long long k = key[c];
    const unsigned low = (unsigned)k;
    winner[c] = (low == 0xFFFFFFFFu) ? -1 : (int)(0xFFFFFFFEu - low);
    if (low != 0xFFFFFFFFu) map_value[c] = unordered_f32((unsigned)(k >> 32));
}

}  // namespace flb

// =======================================================================================
// IKFoM-typed update (SURVEY.md section 8 row a8): esekfom update_iterated_dyn_share_modified
// (include/IKFoM_toolkit/esekfom/esekfom.hpp:1619-1928) driven by h_share_model
// (src/laserMapping.cpp:960-1094), 23-DoF state_ikfom, all on the device in one launch.
// =======================================================================================
namespace flb {

struct IkfomCtrl {
    int i;            // loop index of esekfom.hpp:1633 (starts at -1)
    int t;            // convergence counter (:1824)
    int converge;     // dyn_share.converge: the NEXT pass redoes the kNN (:994 of laserMapping.cpp)
    int stop;
    int passes, knn_passes, n_eff_last, converged_last, status;
    double res_mean_last;
    long long rows_total;
};

struct IkfomParamsDev {
    double R;
    int max_iteration;
    double limit[kIk];
};

struct IkfomSolveArgs {
    StateIkfom* state;             // x_ and P_ (in / out)
    const StateIkfom* state_prop;  // x_propagated and P_propagated
    IkfomCtrl* ctrl;
    const double* partials;        // nblocks * lio_packed(12)
    int nblocks;
    IkfomParamsDev prm;
};

struct IkLeaderSmem {
    StateIkfom x;                  // head = x_, P = the working P_
    double xp_head[kIkHead];
    double L[kIk * kIk];
    double Kx[kIk * 12];
    double K[kIk * 12];            // P_inv[:, :12]
    double HTH[144], HTh[12];
    double S[12 * 25];             // 12 x 24 Gauss-Jordan workspace, row stride 25
    double P11inv[144];
    double B[11 * 12];
    double dx[kIk], dx_new[kIk], dxo[kIk], Kh[kIk];
    double AT[2][9], T2[4];
    double packed[96];
    int flags[4];
};

// Gauss-Jordan of an N x 2N system (row stride LD) by the whole block, no pivoting (SPD).
template <int N, int LD, int NT>
__device__ __forceinline__ void gj_block(double* S, int* bad, int tid) {
    constexpr int COLS = 2 * N, E = N * COLS, PER = (E + NT - 1) / NT;
    for (int k = 0; k < N; ++k) {
        const double piv = S[k * LD + k];
        if (!(fabs(piv) > 1e-300) || !isfinite(piv)) *bad = 1;
        const double inv = __drcp_rn(piv);
        double v[PER];
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const int e = tid + q * NT;
            if (e < E) {
                const int i = e / COLS, j = e - i * COLS;
                const double rkj = S[k * LD + j] * inv;
                v[q] = (i == k) ? rkj : S[i * LD + j] - S[i * LD + k] * rkj;
            }
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const int e = tid + q * NT;
            if (e < E) {
                const int i = e / COLS, j = e - i * COLS;
                S[i * LD + j] = v[q];
            }
        }
        __syncthreads();
    }
}

// M[idx.., c] = T * src[idx.., c] for every column c (T is KxK); threads c < cols.
template <int KD>
__device__ __forceinline__ void ik_rows_apply(double* M, int ldm, int cols, int idx, const double* T, const double* src,
                                              int lds, int tid) {
    if (tid < cols) {
        double v[KD];
#pragma unroll
        for (int i = 0; i < KD; ++i) {
            double s = 0;
#pragma unroll
            for (int k = 0; k < KD; ++k) s += T[i * KD + k] * src[(idx + k) * lds + tid];
            v[i] = s;
        }
#pragma unroll
        for (int i = 0; i < KD; ++i) M[(idx + i) * ldm + tid] = v[i];
    }
}
// M[r, idx..] = M[r, idx..] * T^T for every row r; threads r < kIk.
template <int KD>
__device__ __forceinline__ void ik_cols_apply_T(double* M, int idx, const double* T, int tid) {
    if (tid < kIk) {
        double v[KD];
#pragma unroll
        for (int j = 0; j < KD; ++j) {
            double s = 0;
#pragma unroll
            for (int k = 0; k < KD; ++k) s += M[tid * kIk + idx + k] * T[j * KD + k];
            v[j] = s;
        }
#pragma unroll
        for (int j = 0; j < KD; ++j) M[tid * kIk + idx + j] = v[j];
    }
}

template <int NT>
__device__ __forceinline__ void ikfom_leader(const IkfomSolveArgs& s, IkLeaderSmem& sm, bool first, int it, int tcount,
                                             int converge_in) {
    constexpr int K = lio_packed(12);
    const int tid = threadIdx.x;
    // ---- loads: x_ head, x_propagated head, P_ = P_propagated (:1654)
    {
        const double* xs = reinterpret_cast<const double*>(s.state);
        const double* ps = reinterpret_cast<const double*>(s.state_prop);
        if (tid < kIkHead) reinterpret_cast<double*>(&sm.x)[tid] = __ldcg(xs + tid);
        else if (tid < 2 * kIkHead) sm.xp_head[tid - kIkHead] = __ldcg(ps + tid - kIkHead);
        constexpr int PER = (kIk * kIk + NT - 1) / NT;
        double v[PER];
#pragma unroll
        for (int u = 0; u < PER; ++u) { const int e = tid + u * NT; v[u] = e < kIk * kIk ? __ldcg(ps + kIkHead + e) : 0.0; }
#pragma unroll
        for (int u = 0; u < PER; ++u) { const int e = tid + u * NT; if (e < kIk * kIk) sm.x.P[e] = v[u]; }
    }
    // ---- fixed-order reduction of the block partials (block order, 16 loads in flight)
    if (tid < K) {
        double acc = 0.0;
        for (int b = 0; b < s.nblocks; b += 16) {
            double v[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) v[u] = (b + u < s.nblocks) ? __ldcg(s.partials + (size_t)(b + u) * K + tid) : 0.0;
#pragma unroll
            for (int u = 0; u < 16; ++u) acc += v[u];
        }
        sm.packed[tid] = acc;
    }
    if (tid == 0) sm.flags[3] = 0;
    __syncthreads();
    if (tid == 0) {   // HTH (12x12 symmetric) and h_x^T h
        int k = 0;
        for (int r = 0; r < 12; ++r)
            for (int c = r; c < 12; ++c) { sm.HTH[r * 12 + c] = sm.packed[k]; sm.HTH[c * 12 + r] = sm.packed[k]; ++k; }
        for (int r = 0; r < 12; ++r) sm.HTh[r] = sm.packed[78 + r];
    }
    if (tid == 32) {  // dx = x_ [-] x_propagated (:1646) and the projection matrices (:1656-1696)
        StateIkfom* xp = reinterpret_cast<StateIkfom*>(sm.xp_head);   // head only
        ikfom_boxminus(sm.x, *xp, sm.dx);
        for (int a = 0; a < kIk; ++a) sm.dx_new[a] = sm.dx[a];
        for (int q = 0; q < 2; ++q) {
            const int idx = 3 + 3 * q;
            double A[9], v[3];
            mtk_A_matrix(sm.dx + idx, A);
            transpose_small(A, 3, 3, sm.AT[q]);
            mm_small(sm.AT[q], 3, 3, sm.dx_new + idx, 1, v);
            for (int a = 0; a < 3; ++a) sm.dx_new[idx + a] = v[a];
        }
        double Nx[6], Mx[6], v2[2];
        s2_Nx_yy(sm.x.grav, Nx);
        s2_Mx(xp->grav, sm.dx + 21, Mx);
        mm_small(Nx, 2, 3, Mx, 2, sm.T2);
        mm_small(sm.T2, 2, 2, sm.dx_new + 21, 1, v2);
        sm.dx_new[21] = v2[0];
        sm.dx_new[22] = v2[1];
    }
    __syncthreads();
    double* P = sm.x.P;
    for (int q = 0; q < 2; ++q) {
        ik_rows_apply<3>(P, kIk, kIk, 3 + 3 * q, sm.AT[q], P, kIk, tid);
        __syncthreads();
        ik_cols_apply_T<3>(P, 3 + 3 * q, sm.AT[q], tid);
        __syncthreads();
    }
    ik_rows_apply<2>(P, kIk, kIk, 21, sm.T2, P, kIk, tid);
    __syncthreads();
    ik_cols_apply_T<2>(P, 21, sm.T2, tid);
    __syncthreads();
    // ---- P_inv[:, :12] by the Schur complement (see the 18-DoF leader): P11 = P_[:12, :12]
    for (int e = tid; e < 12 * 24; e += NT) {
        const int i = e / 24, j = e - i * 24;
        sm.S[i * 25 + j] = (j < 12) ? P[i * kIk + j] : ((j - 12 == i) ? 1.0 : 0.0);
    }
    __syncthreads();
    gj_block<12, 25, NT>(sm.S, &sm.flags[3], tid);
    for (int e = tid; e < 144; e += NT) sm.P11inv[e] = sm.S[(e / 12) * 25 + 12 + (e % 12)];
    __syncthreads();
    for (int e = tid; e < 11 * 12; e += NT) {   // B = P21 * P11^-1
        const int i = e / 12, j = e - i * 12;
        double acc = 0;
#pragma unroll
        for (int k = 0; k < 12; ++k) acc += P[(12 + i) * kIk + k] * sm.P11inv[k * 12 + j];
        sm.B[e] = acc;
    }
    for (int e = tid; e < 12 * 24; e += NT) {
        const int i = e / 24, j = e - i * 24;
        sm.S[i * 25 + j] = (j < 12) ? sm.HTH[i * 12 + j] + s.prm.R * sm.P11inv[i * 12 + j] : ((j - 12 == i) ? 1.0 : 0.0);
    }
    __syncthreads();
    gj_block<12, 25, NT>(sm.S, &sm.flags[3], tid);
    for (int e = tid; e < 144; e += NT) sm.K[e] = sm.S[(e / 12) * 25 + 12 + (e % 12)];   // Kt
    __syncthreads();
    for (int e = tid; e < 11 * 12; e += NT) {   // Kb = B * Kt
        const int i = e / 12, j = e - i * 12;
        double acc = 0;
#pragma unroll
        for (int k = 0; k < 12; ++k) acc += sm.B[i * 12 + k] * sm.K[k * 12 + j];
        sm.K[144 + e] = acc;
    }
    __syncthreads();
    for (int e = tid; e < kIk * 12; e += NT) {  // K_x[:, :12] = P_inv[:, :12] * HTH   (:1806)
        const int i = e / 12, j = e - i * 12;
        double acc = 0;
#pragma unroll
        for (int k = 0; k < 12; ++k) acc += sm.K[i * 12 + k] * sm.HTH[k * 12 + j];
        sm.Kx[e] = acc;
    }
    if (tid < kIk) {                            // K_h = P_inv[:, :12] * h_x^T h       (:1801)
        double acc = 0;
#pragma unroll
        for (int k = 0; k < 12; ++k) acc += sm.K[tid * 12 + k] * sm.HTh[k];
        sm.Kh[tid] = acc;
    }
    __syncthreads();
    if (tid < kIk) {                            // dx_ = K_h + (K_x - I) * dx_new      (:1812)
        double acc = sm.Kh[tid];
#pragma unroll
        for (int k = 0; k < 12; ++k) acc += sm.Kx[tid * 12 + k] * sm.dx_new[k];
        sm.dxo[tid] = acc - sm.dx_new[tid];
    }
    __syncthreads();
    if (tid == 0) {
        IkfomCtrl c;
        if (first) {
            c.passes = c.knn_passes = 0;
            c.rows_total = 0;
            c.status = 0;
        } else {
            c.passes = __ldcg(&s.ctrl->passes);
            c.knn_passes = __ldcg(&s.ctrl->knn_passes);
            c.rows_total = __ldcg(&s.ctrl->rows_total);
            c.status = __ldcg(&s.ctrl->status);
        }
        const bool ok = sm.flags[3] == 0;
        const int n_eff = (int)sm.packed[K - 2];
        c.passes += 1;
        c.knn_passes += converge_in ? 1 : 0;
        c.n_eff_last = n_eff;
        c.res_mean_last = sm.packed[K - 1] / (double)n_eff;
        c.rows_total += n_eff;
        ikfom_boxplus(sm.x, sm.dxo);                                   // :1814
        int conv = 1;
        for (int a = 0; a < kIk; ++a)
            if (fabs(sm.dxo[a]) > s.prm.limit[a]) { conv = 0; break; } // :1816-1823
        int t = tcount;
        if (conv) t++;
        if (!t && it == s.prm.max_iteration - 2) conv = 1;             // :1826-1829
        int fin = (t > 1 || it == s.prm.max_iteration - 1) ? 1 : 0;    // :1831
        if (!ok) { fin = 1; c.status = -5; }
        c.converged_last = conv;
        c.i = it + 1;
        c.t = t;
        c.converge = conv;
        c.stop = fin;
        *s.ctrl = c;
        sm.flags[0] = fin && ok;
        if (fin && ok) {                                               // projections with dx_ (:1836-1893)
            for (int q = 0; q < 2; ++q) {
                double A[9];
                mtk_A_matrix(sm.dxo + 3 + 3 * q, A);
                transpose_small(A, 3, 3, sm.AT[q]);
            }
            double Nx[6], Mx[6];
            s2_Nx_yy(sm.x.grav, Nx);
            s2_Mx(reinterpret_cast<StateIkfom*>(sm.xp_head)->grav, sm.dxo + 21, Mx);
            mm_small(Nx, 2, 3, Mx, 2, sm.T2);
        }
    }
    __syncthreads();
    if (sm.flags[0]) {
        for (int e = tid; e < kIk * kIk; e += NT) sm.L[e] = P[e];      // L_ = P_ (:1833)
        __syncthreads();
        for (int q = 0; q < 2; ++q) {
            const int idx = 3 + 3 * q;
            ik_rows_apply<3>(sm.L, kIk, kIk, idx, sm.AT[q], P, kIk, tid);        // L_ rows from P_ rows
            if (tid >= 32 && tid < 44) ik_rows_apply<3>(sm.Kx, 12, 12, idx, sm.AT[q], sm.Kx, 12, tid - 32);
            __syncthreads();
            ik_cols_apply_T<3>(sm.L, idx, sm.AT[q], tid);
            if (tid >= 32 && tid < 32 + kIk) ik_cols_apply_T<3>(P, idx, sm.AT[q], tid - 32);
            __syncthreads();
        }
        ik_rows_apply<2>(sm.L, kIk, kIk, 21, sm.T2, P, kIk, tid);
        if (tid >= 32 && tid < 44) ik_rows_apply<2>(sm.Kx, 12, 12, 21, sm.T2, sm.Kx, 12, tid - 32);
        __syncthreads();
        ik_cols_apply_T<2>(sm.L, 21, sm.T2, tid);
        if (tid >= 32 && tid < 32 + kIk) ik_cols_apply_T<2>(P, 21, sm.T2, tid - 32);
        __syncthreads();
        // P_ = L_ - K_x[:, :12] * P_[:12, :]   (:1918)
        double* Pg = s.state->P;
        for (int e = tid; e < kIk * kIk; e += NT) {
            const int i = e / kIk, j = e - i * kIk;
            double acc = 0;
#pragma unroll
            for (int k = 0; k < 12; ++k) acc += sm.Kx[i * 12 + k] * P[k * kIk + j];
            Pg[e] = sm.L[e] - acc;
        }
    }
    if (tid < kIkHead) reinterpret_cast<double*>(s.state)[tid] = reinterpret_cast<const double*>(&sm.x)[tid];
}

// Pose of a pass from state_ikfom: R = rot.toRotationMatrix(), extrinsic from offset_R_L_I / offset_T_L_I
__device__ __forceinline__ void ikfom_make_pose(const StateIkfom* st, LioPose& pose) {
    double head[kIkHead];
    const double* g = reinterpret_cast<const double*>(st);
    for (int i = 0; i < kIkHead; ++i) head[i] = __ldcg(g + i);
    const StateIkfom* x = reinterpret_cast<const StateIkfom*>(head);
    quat_to_R(x->rot, pose.R);
    quat_to_R(x->offset_R_L_I, pose.R_LI);
    for (int i = 0; i < 3; ++i) { pose.p[i] = x->pos[i]; pose.t_LI[i] = x->offset_T_L_I[i]; }
    m3_T(pose.R, pose.Rt);
    m3_T(pose.R_LI, pose.RLIt);
}

template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) k_lio_update_ikfom_persistent(LioArgs a, IkfomSolveArgs s, GridBarrier* bar) {
    constexpr int K = lio_packed(12);
    __shared__ LioPose s_pose;
    __shared__ double s_acc[BLOCK / 32][K];
    __shared__ unsigned s_bar[2];
    __shared__ IkLeaderSmem sm;
    __shared__ int s_rows[18][BLOCK];
    const int tid = threadIdx.x;
    int it = -1, tcount = 0, converge = 1;     // esekfom.hpp:1622-1624, :1633
    bool first = true;
    for (;;) {
        if (tid == 0) ikfom_make_pose(s.state, s_pose);
        __syncthreads();
        double acc[K];
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = 0.0;
        for (int c = (tid >> 5) * gridDim.x + blockIdx.x; c * 32 < a.N; c += (BLOCK / 32) * gridDim.x) {
            const int i = c * 32 + (tid & 31);
            if (i < a.N) {
                bool active;
                double row[12], z, absres;
                lio_point<12>(a, s_pose, converge != 0, i, active, row, z, absres, &s_rows[0][tid], BLOCK);   // converge => redo kNN (:994)
                if (active) lio_accumulate<12>(acc, row, z, absres);
            }
        }
        block_reduce_store<K, BLOCK>(acc, s_acc, a.partials);
        const bool leader = grid_arrive(bar, gridDim.x, s_bar);
        if (leader) {
            ikfom_leader<BLOCK>(s, sm, first, it, tcount, converge);
            grid_release(bar, s_bar);
        } else {
            if (!grid_wait(bar, s_bar)) return;
        }
        const int stop = __ldcg(&s.ctrl->stop);
        converge = __ldcg(&s.ctrl->converge);
        tcount = __ldcg(&s.ctrl->t);
        it = __ldcg(&s.ctrl->i);
        first = false;
        if (stop) break;
    }
}

}  // namespace flb
