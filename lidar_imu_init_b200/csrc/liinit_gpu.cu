// liinit_gpu.cu -- C-ABI implementation (include/liinit_gpu.h) over the sm_100a kernels.
//
// One context = one GPU, one stream, one device-resident map, one resident scan. No CPU fallback:
// every entry point fails with LIINIT_ERR_CUDA if the CUDA runtime reports an error.
#include "../../include/liinit_gpu.h"

#include <cuda_runtime.h>
#ifndef LI_SIMT_EMUL
#include <dlfcn.h>
#include <nccl.h>   // types only: the library is dlopen()ed when a communicator is asked for (no link-time dependency)
#endif

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"
#include "icp_kernels.cuh"
#include "knn_kernels.cuh"
#include "knn_general.cuh"
#include "cells.cuh"
#include "map_kernels.cuh"
#include "voxelgrid_kernels.cuh"
#include "undistort_kernels.cuh"

#ifndef LI_CELLS_MINB
#define LI_CELLS_MINB 6
#endif
#ifndef LIINIT_KNN_DEFAULT
#define LIINIT_KNN_DEFAULT LIINIT_KNN_BRICKS   // what knn_index = 0 selects
#endif


namespace {

thread_local std::string g_create_error;

#ifndef LI_SIMT_EMUL
// NCCL entry points, resolved at run time from libnccl.so.2 (the copy the process already has -- e.g. the one a PyTorch host
// application loaded -- or the system one). A single-GPU deployment never touches it.
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string err;
};
NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (tried) return api.lib ? &api : nullptr;
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
        api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (api.lib) break;
    }
    if (!api.lib) {
        api.err = std::string("dlopen(libnccl.so.2): ") + dlerror();
        return nullptr;
    }
    bool ok = true;
    auto sym = [&](const char* n) { void* f = dlsym(api.lib, n); if (!f) { ok = false; api.err = std::string("missing NCCL symbol ") + n; } return f; };
    api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
    api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
    api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
    api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
    api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
    if (!ok) {
        dlclose(api.lib);
        api.lib = nullptr;
        return nullptr;
    }
    return &api;
}
#endif

// device scratch (per call, or owned by the context) that is released on every return path (the CU() macro returns early on a CUDA error)
template <class T>
struct DevBuf {
    T* p = nullptr;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t count) { return cudaMalloc(&p, count * sizeof(T)); }
};

struct Ctx {
    liinit_config cfg;
    int device = 0;
    int num_sms = 148;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evm = nullptr;
    bool last_was_search = false;
    std::string err;

    // map
    MapDev M{};
    unsigned hash_slots = 0;
    int* d_counters = nullptr;
    int* h_counters = nullptr;   // pinned
    unsigned long long* h_pool_top = nullptr;   // pinned: the bump allocator's value after the last map update
    // staging
    float* d_stage_raw = nullptr;   // strided host layout
    size_t stage_raw_floats = 0;
    float4* d_stage_pts = nullptr;  // repacked batch
    int stage_pts_cap = 0;
    int* d_slot_of = nullptr;
    int* d_vslot_of = nullptr;
    int* d_flag = nullptr;
    int* d_ins = nullptr;
    int* d_vg_imin = nullptr;      // voxel-grid: first point index per leaf
    int* d_vg_block = nullptr;     // (unused scratch)
    unsigned* d_rs_keys = nullptr;  // radix sort ping-pong buffers + histogram
    unsigned* d_rs_vals = nullptr;
    int* d_rs_hist = nullptr;
    int* d_vg_misc = nullptr;      // [0..5] min/max (ordered ints), [6] out count, [7] error bits
    VgParams* d_vg_params = nullptr;
    int raw_n = 0;                          // raw (not yet downsampled) cloud staged in d_stage_pts, w = time [ms]
    unsigned long long* d_tmin_idx = nullptr;
    double* d_poses = nullptr;              // IMU pose table for the undistortion (<= 4096 x 22 doubles)
    VoxTmp V{};
    // scan
    ScanDev S{};
    float4* d_body = nullptr;
    float4* d_world = nullptr;
    int* d_near_ids = nullptr;
    float4* d_near_xyz = nullptr;
    unsigned char* d_selected = nullptr;
    float4* d_normvec = nullptr;
    int scan_n = 0;                // points of the resident scan (the whole frame)
    // multi-GPU (SURVEY.md section 8e): the map is replicated, every rank holds the whole frame and PROCESSES the shard
    // [shard_lo, shard_lo + S.n) of it; one all-reduce of the 160-double block per pass, inside liinit_icp_iterate*
    int nranks = 1, rank = 0;
    int shard_lo = 0;
#ifndef LI_SIMT_EMUL
    ncclComm_t comm = nullptr;
#endif
    double* d_acc = nullptr;       // the rank's own accumulator block (N > 1) ...
    double* d_red = nullptr;       // ... and its sum over the ranks (NCCL mode)
    // peer-memory mode (default when CUDA IPC between the ranks works): the sum happens in the last block of the plane kernel
    bool comm_p2p = false;
    void* d_xbuf = nullptr;        // this rank's exchange buffer: [2][nranks][160] doubles + [2][nranks] flags
    XchgTable* d_xtab = nullptr;   // every rank's buffer as mapped into this process
    void* peer_map[LI_MAX_RANKS] = {nullptr};   // what cudaIpcOpenMemHandle returned (closed in liinit_destroy)
    unsigned xseq = 0;             // pass sequence number (identical on every rank: the passes are collective)
    bool state_gathered = true;    // per-point results of the other ranks' shards are present on this device
    unsigned map_epoch = 0;        // bumped by everything that can REMOVE a map point (Build, downsample inserts, box delete, compaction)
    unsigned nbr_epoch = 0;        // map_epoch when the resident scan's Nearest_Points were found
    bool reseed = true;            // later search passes of a scan start from the previous pass's neighbours (liinit_set_reseed)
    bool have_neighbors = false;   // a search pass has filled near_xyz for the resident scan (point copies: map updates do not invalidate them)
    bool scan_fresh = false;   // new scan whose flags / neighbour lists have not been initialised yet (see init_scan_state)
    const float* attached = nullptr;   // device alias of a page-locked host scan not copied yet (liinit_scan_attach_host)
    int attached_stride = 0;
    bool attached_slot_done = false;   // N > 1: this rank's slot has been pulled in by its search kernel, the other slots are still on the host
    // reduction
    double* d_partials = nullptr;
    unsigned* d_done = nullptr;
    double* h_out = nullptr;    // pinned + mapped 160
    double* h_out_dev = nullptr;   // its device alias
    int max_blocks = 0;
    // knn query scratch
    float* d_q_d2 = nullptr;
    // k-NN search for any k / max_dist (knn_general.cuh): copies of the map's brick entries, walked by far / unbounded queries;
    // rebuilt on the stream when map_version moved since
    unsigned map_version = 0;      // bumped by every call that changes the map
    DevBuf<uint4> knn_occ;         // [hash_slots] (a brick per hash slot at most), allocated on first use
    unsigned knn_occ_version = 0;
    bool knn_occ_valid = false;
    // stats
    long long launches = 0;
    float last_ms = 0.f;
    int last_launches = 0;
    int group = 4;
    int cells_search = LI_CELLS_SEARCH_DEFAULT;   // 1 shells on cells, 2 growing boxes, 3 growing boxes enumerate + stream (developer A/B: LIINIT_CELLS_SEARCH)
    bool cells_dynamic = false;       // cells search kernel with warp-granular dynamic scheduling (LIINIT_CELLS_SCHED=dynamic; not yet GPU-measured)
    unsigned* d_ticket = nullptr;
    bool cells_refresh_warp = true;   // directory refresh: warp per brick (false: thread per brick, the version the CPU checker runs)
    bool cells = false;   // knn_index = LIINIT_KNN_CELLS: per-brick cell directory + thread-per-point search (cells.cuh)
    float rho2 = 0.09f;   // squared seed radius of the 5-NN search
};

#define CU(call)                                                                                     \
    do {                                                                                             \
        cudaError_t _e = (call);                                                                     \
        if (_e != cudaSuccess) {                                                                     \
            c->err = std::string(#call) + ": " + cudaGetErrorString(_e);                             \
            return LIINIT_ERR_CUDA;                                                                  \
        }                                                                                            \
    } while (0)

inline int nblk(long long n, int t) { return (int)((n + t - 1) / t); }

int fail(Ctx* c, int code, const std::string& msg) {
    c->err = msg;
    return code;
}

// copy n points with a float stride from host to d_stage_pts[0..n) as float4
int stage_points(Ctx* c, const float* xyz, int stride, int n) {
    if (n > c->stage_pts_cap) return fail(c, LIINIT_ERR_CAPACITY, "batch exceeds staging capacity");
    c->raw_n = 0;   // the staging buffer is shared with the raw-scan front end
    if (stride == 4) {
        CU(cudaMemcpyAsync(c->d_stage_pts, xyz, (size_t)n * 16, cudaMemcpyHostToDevice, c->stream));
        return LIINIT_OK;
    }
    if (stride != 3 && stride != 12) return fail(c, LIINIT_ERR_INVALID, "stride_floats must be 3, 4 or 12");
    size_t nf = (size_t)n * stride;
    if (nf > c->stage_raw_floats) return fail(c, LIINIT_ERR_CAPACITY, "batch exceeds raw staging capacity");
    CU(cudaMemcpyAsync(c->d_stage_raw, xyz, nf * 4, cudaMemcpyHostToDevice, c->stream));
    k_repack<<<nblk(n, 256), 256, 0, c->stream>>>(c->d_stage_raw, stride, n, c->d_stage_pts);
    c->launches++;
    CU(cudaGetLastError());
    return LIINIT_OK;
}

int fetch_counters(Ctx* c) {
    CU(cudaMemcpyAsync(c->h_counters, c->d_counters, sizeof(int) * CNT_COUNT, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(c->h_pool_top, c->M.pool_top, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return LIINIT_OK;
}

// Capacity errors are reported ONCE, to the call that hit them: the bits are cleared on the device so that the calls after a box
// delete / a compaction are judged on their own (they used to stay set until the next Build).
int check_map_err(Ctx* c) {
    int e = c->h_counters[CNT_ERR];
    if (e & (ERR_HASH_FULL | ERR_POOL_FULL)) {
        cudaMemsetAsync(c->d_counters + CNT_ERR, 0, sizeof(int), c->stream);
        c->h_counters[CNT_ERR] = 0;
    }
    if (e & ERR_POOL_FULL) {
        // the failed reservations left the bump allocator beyond the capacity (k_ins_reserve): back to the end of the last slab in use
        const int nb = c->h_counters[CNT_BRICKS];
        cudaMemsetAsync(c->M.pool_top, 0, sizeof(unsigned long long), c->stream);
        if (nb > 0) {
            k_pool_top_recompute<<<nblk(nb, 256), 256, 0, c->stream>>>(c->M, nb);
            c->launches++;
        }
        cudaMemcpyAsync(c->h_pool_top, c->M.pool_top, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream);
        cudaStreamSynchronize(c->stream);
    }
    if (e & ERR_HASH_FULL) return fail(c, LIINIT_ERR_CAPACITY, "brick hash table full (raise hash_capacity_log2 / max_map_points)");
    if (e & ERR_POOL_FULL) return fail(c, LIINIT_ERR_CAPACITY, "map point pool full (raise max_map_points, or liinit_map_compact after deletes)");
    return LIINIT_OK;
}

int reset_batch_counters(Ctx* c) {
    // touched, changed, nadd, nnod reset; err, live, bricks, dropped persist
    static const int zeros[CNT_COUNT] = {0};
    CU(cudaMemcpyAsync(c->d_counters + CNT_TOUCHED, zeros, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->d_counters + CNT_CHANGED, zeros, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->d_counters + CNT_COUPLED, zeros, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    return LIINIT_OK;
}

// cell directory of the bricks the batch touched (after the commit / compaction that fixed their counts)
void refresh_cells_touched(Ctx* c) {
    if (!c->cells) return;
    if (c->cells_refresh_warp) k_cells_refresh_touched_warp<<<c->num_sms * 16, 128, 0, c->stream>>>(c->M);
    else k_cells_refresh_touched<<<c->num_sms * 8, 128, 0, c->stream>>>(c->M);
    c->launches++;
}

// plain insert of pts[0..n) (optionally only flag==want)
int plain_insert(Ctx* c, const float4* pts, int n, const int* sel, int want) {
    if (n <= 0) return LIINIT_OK;
    int r = reset_batch_counters(c);
    if (r) return r;
    k_ins_count<<<nblk(n, 256), 256, 0, c->stream>>>(c->M, pts, n, sel, want, c->d_slot_of);
    // the number of touched bricks is only known on the device: fixed grids, grid-stride loops inside
    const int gfix = c->num_sms * 8;
    k_ins_reserve<<<gfix, 256, 0, c->stream>>>(c->M);
    k_ins_append<<<nblk(n, 256), 256, 0, c->stream>>>(c->M, pts, n, c->d_slot_of);
    k_ins_commit<<<gfix, 256, 0, c->stream>>>(c->M);
    c->launches += 4;
    refresh_cells_touched(c);
    CU(cudaGetLastError());
    return LIINIT_OK;
}

// the temporary voxel hash, shrunk to the next power of two >= 2n slots (never beyond the allocation)
VoxTmp sized_vox(Ctx* c, int n) {
    VoxTmp V = c->V;
    unsigned m = 1024;
    while (m < 2u * (unsigned)n && m - 1 < c->V.mask) m <<= 1;
    if (m - 1 < V.mask) V.mask = m - 1;
    return V;
}

int downsample_insert(Ctx* c, const float4* pts, int n, const int* sel, int want) {
    if (n <= 0) return LIINIT_OK;
    int r = reset_batch_counters(c);
    if (r) return r;
    VoxTmp V = sized_vox(c, n);   // batch-sized temporary hash: clearing / walking 2M slots for a 10k-point batch is waste
    k_vox_clear<<<nblk((long long)V.mask + 1, 256), 256, 0, c->stream>>>(V);
    k_ds_link<<<nblk(n, 256), 256, 0, c->stream>>>(c->M, V, pts, n, sel, want, c->d_vslot_of, c->d_slot_of, c->d_ins);
    k_ins_reserve<<<c->num_sms * 8, 256, 0, c->stream>>>(c->M);
    k_ds_scan<<<nblk((long long)V.mask + 1, 128), 128, 0, c->stream>>>(c->M, V, pts, c->d_vslot_of);
    k_ds_replay<<<nblk((long long)V.mask + 1, 128), 128, 0, c->stream>>>(c->M, V, pts, c->d_vslot_of, c->d_ins);
    // boxes that share a point with another box of the batch (one-ulp overlaps of the float boxes): one warp, batch order (returns at once when there are none)
    k_ds_coupled<<<1, 32, 0, c->stream>>>(c->M, V, pts, c->d_vslot_of, c->d_ins, reinterpret_cast<int*>(c->d_rs_keys), reinterpret_cast<int*>(c->d_rs_vals));
    k_ds_append<<<nblk(n, 256), 256, 0, c->stream>>>(c->M, pts, n, c->d_slot_of, c->d_ins);
    // tombstoned bricks were added to the touched list by the replay (worst case n + n bricks): grid-stride inside
    k_ds_compact<<<c->num_sms * 8, 256, 0, c->stream>>>(c->M);
    c->launches += 8;
    refresh_cells_touched(c);
    CU(cudaGetLastError());
    return LIINIT_OK;
}

void fill_pose(PoseD& P, const double* R, const double* p, const double* RLI, const double* TLI) {
    memcpy(P.R, R, 72);
    memcpy(P.p, p, 24);
    memcpy(P.RLI, RLI, 72);
    memcpy(P.TLI, TLI, 24);
}

// An attached host scan that something other than the search kernel needs: pull it into d_body now.
void materialize_scan(Ctx* c) {
    if (!c->attached) return;
    if (c->attached_slot_done) {   // only what the search kernel did not read: the other ranks' slots [0, lo) and [lo + S.n, n)
        const int lo = c->shard_lo, hi = c->shard_lo + c->S.n;
        if (lo > 0) {
            k_repack<<<nblk(lo, 256), 256, 0, c->stream>>>(c->attached, c->attached_stride, lo, c->d_body);
            c->launches++;
        }
        if (hi < c->scan_n) {
            k_repack<<<nblk(c->scan_n - hi, 256), 256, 0, c->stream>>>(c->attached + (size_t)hi * c->attached_stride, c->attached_stride, c->scan_n - hi,
                                                                       c->d_body + hi);
            c->launches++;
        }
    } else {
        k_repack<<<nblk(c->scan_n, 256), 256, 0, c->stream>>>(c->attached, c->attached_stride, c->scan_n, c->d_body);
        c->launches++;
    }
    c->attached = nullptr;
    c->attached_slot_done = false;
}

// A new scan starts with nothing selected and no neighbours (Nearest_Points / point_selected_surf at iteration 0). The search
// pass that normally follows overwrites both arrays for every point of the scan, so the two fills are only issued when
// something else looks at them first (map_incremental, the download hooks): two stream operations fewer per scan.
int init_scan_state(Ctx* c) {
    if (!c->scan_fresh) return LIINIT_OK;
    CU(cudaMemsetAsync(c->d_selected, 0, (size_t)c->scan_n, c->stream));
    CU(cudaMemsetAsync(c->d_near_xyz, 0, (size_t)c->scan_n * 5 * sizeof(float4), c->stream));   // w = 0: no neighbour at any rank
    c->scan_fresh = false;
    return LIINIT_OK;
}

// A new frame of n points is resident (or attached): this rank's shard is [rank * cnt, rank * cnt + cnt) clipped to n with
// cnt = ceil(n / nranks) -- equal-sized slots, so that the per-point results can be all-gathered in place.
void set_scan(Ctx* c, int n) {
    c->scan_n = n;
    const int cnt = (n + c->nranks - 1) / c->nranks;
    int lo = c->rank * cnt;
    if (lo > n) lo = n;
    int hi = lo + cnt;
    if (hi > n) hi = n;
    c->shard_lo = lo;
    c->S.body = c->d_body + lo;
    c->S.world = c->d_world + lo;
    c->S.near_ids = c->d_near_ids + (size_t)lo * 5;
    c->S.near_xyz = c->d_near_xyz + (size_t)lo * 5;
    c->S.selected = c->d_selected + lo;
    c->S.normvec = c->d_normvec + lo;
    c->S.n = hi - lo;
    c->have_neighbors = false;
    c->scan_fresh = true;
    c->state_gathered = c->nranks == 1;
}

// Lanes per scan point when the caller left knn_group_lanes = 0. A warp works on 32/G points at once and lives as long as its slowest
// one: 4 lanes give the best throughput once every SM holds several such batches, but a small frame then occupies a fraction of the
// GPU for a long batch time. Measured on one B200 (C2 scene, both poses; profiles/r02/probe_frame_size_vs_group_lanes.log for the first
// shape of the search, profiles/r02/probe_v3_parameters_and_frame_sizes.log for the present one), search kernel ms at the initial pose:
//   8k points: 0.044 (G = 4) / 0.029 (8) / 0.023 (16) / 0.023 (32);   20k: 0.044 / 0.033 / 0.036 / 0.040;   45k: 0.058 / 0.049 / 0.062 / 0.082;
//   60k: 0.067 / 0.068;   90k: 0.084 / 0.088;   130k: 0.109 / 0.111;   170k: 0.129 / 0.147;   240k: 0.161 / 0.190.
int group_for(int n) {
    if (n <= 14000) return 32;
    if (n <= 70000) return 8;
    return 4;
}

// The search kernel of a pass reads an attached host frame in place: its own slot only. With one rank that is the whole frame and
// nothing is left to copy; with several the rest stays on the host until somebody needs the whole frame (materialize_scan).
const float* attached_slot(Ctx* c) {
    return (c->attached && !c->attached_slot_done) ? c->attached + (size_t)c->shard_lo * c->attached_stride : nullptr;
}
void attached_slot_read(Ctx* c) {
    if (c->nranks > 1 && c->S.n < c->scan_n) c->attached_slot_done = true;
    else c->attached = nullptr;
}

template <int G>
void launch_knn_scan(Ctx* c, const PoseD& P) {
    long long threads = (long long)c->S.n * G;
    int grid = nblk(threads, LI_KNN_THREADS);
    int cap = c->max_blocks * (256 / LI_KNN_THREADS);
    if (grid > cap) grid = cap;
    // a later search pass of the same scan, no map point removed in between: seeded by the previous pass's neighbours (knn_kernels.cuh)
    const bool seeded = c->have_neighbors && !c->scan_fresh && c->nbr_epoch == c->map_epoch && c->reseed;
    if (const float* raw = attached_slot(c)) {
        k_knn_scan<G, true><<<grid, LI_KNN_THREADS, 0, c->stream>>>(c->M, c->S, P, c->rho2, raw, c->attached_stride);
        attached_slot_read(c);   // the kernel leaves the packed copy in d_body
    } else if (seeded) {
        k_knn_scan<G, false, true><<<grid, LI_KNN_THREADS, 0, c->stream>>>(c->M, c->S, P, c->rho2, nullptr, 0);
    } else {
        k_knn_scan<G, false><<<grid, LI_KNN_THREADS, 0, c->stream>>>(c->M, c->S, P, c->rho2, nullptr, 0);
    }
}

#ifndef LI_PLANE_WAVES
#define LI_PLANE_WAVES 1   // the plane pass runs LI_PLANE_WAVES x (2 blocks per SM); each thread strides over the scan
#endif

template <int MINB, int SEARCH>
void launch_knn_cells_scan_t(Ctx* c, const PoseD& P) {
    if (c->cells_dynamic) {   // persistent grid, warps pull 32-point batches from a ticket counter (reset in stream order)
        cudaMemsetAsync(c->d_ticket, 0, sizeof(unsigned), c->stream);
        const int pgrid = c->num_sms * MINB;
        if (const float* raw = attached_slot(c)) {
            k_knn_cells_scan_dyn<true, MINB, SEARCH><<<pgrid, LI_CELLS_THREADS, 0, c->stream>>>(c->M, c->S, P, c->rho2, raw, c->attached_stride, c->d_ticket);
            attached_slot_read(c);
        } else {
            k_knn_cells_scan_dyn<false, MINB, SEARCH><<<pgrid, LI_CELLS_THREADS, 0, c->stream>>>(c->M, c->S, P, c->rho2, nullptr, 0, c->d_ticket);
        }
        return;
    }
    const int grid = nblk(c->S.n, LI_CELLS_THREADS);
    if (const float* raw = attached_slot(c)) {
        k_knn_cells_scan<true, MINB, SEARCH><<<grid, LI_CELLS_THREADS, 0, c->stream>>>(c->M, c->S, P, c->rho2, raw, c->attached_stride);
        attached_slot_read(c);   // the kernel leaves the packed copy in d_body
    } else {
        k_knn_cells_scan<false, MINB, SEARCH><<<grid, LI_CELLS_THREADS, 0, c->stream>>>(c->M, c->S, P, c->rho2, nullptr, 0);
    }
}
// LI_CELLS_MINB (resident blocks per SM the kernel is compiled for): 6 -> 80 registers; measured against 4 (106 registers, no spills)
// and 8 (64 registers, 55 spilled words): 0.56 / 0.60 / 0.72 ms at the initial pose (profiles/r01_cells/ab_stream_final.log)
void launch_knn_cells_scan(Ctx* c, const PoseD& P) {
    if (c->cells_search == 1) launch_knn_cells_scan_t<LI_CELLS_MINB, 1>(c, P);
    else if (c->cells_search == 2) launch_knn_cells_scan_t<LI_CELLS_MINB, 2>(c, P);
    else launch_knn_cells_scan_t<LI_CELLS_MINB, 3>(c, P);
}

template <bool IMU, bool SEARCH>
void launch_plane(Ctx* c, const PoseD& P, double* out) {
    // one wave of 256-thread blocks (2 resident per SM at ~100-130 registers), grid-stride over the scan
    int grid = nblk(c->S.n, 256);
    if (grid > c->num_sms * LI_PLANE_MIN_BLOCKS * LI_PLANE_WAVES) grid = c->num_sms * LI_PLANE_MIN_BLOCKS * LI_PLANE_WAVES;
    if (grid < 1) grid = 1;   // (an empty slot of a multi-GPU frame still takes part in the exchange)
    const XchgTable* X = (c->nranks > 1 && c->comm_p2p) ? c->d_xtab : nullptr;
    // the lockstep search leaves the neighbour copies in S.near_xyz itself; the cell-directory search hands pool offsets over, which
    // the plane kernel of that pass gathers (and leaves as copies); a reuse pass reads the copies
    if (SEARCH && c->cells) k_icp_plane<IMU, SEARCH, true><<<grid, 256, 0, c->stream>>>(c->M, c->S, P, c->d_partials, c->d_done, out, X, c->xseq);
    else k_icp_plane<IMU, SEARCH, false><<<grid, 256, 0, c->stream>>>(c->M, c->S, P, c->d_partials, c->d_done, out, X, c->xseq);
}

// out: where the last block of the plane kernel leaves the 160-double result block -- the caller's device buffer
// (liinit_icp_iterate_device) or the device alias of the context's page-locked host block (liinit_icp_iterate: the
// kernel writes the 1.28 kB over PCIe itself, no copy operation behind it).
int run_pass(Ctx* c, const double* R, const double* p, const double* RLI, const double* TLI, int imu_en, int search, double* out) {
    if (c->scan_n <= 0) return fail(c, LIINIT_ERR_INVALID, "no scan uploaded");
    if (!search && !c->have_neighbors) return fail(c, LIINIT_ERR_INVALID, "reuse pass before any search pass");
    PoseD P;
    fill_pose(P, R, p, RLI, TLI);
    double* const final_out = out;
    if (c->nranks > 1 && !c->comm_p2p) out = c->d_acc;   // NCCL mode: this rank's block; the sum over the ranks goes to final_out below
    if (c->nranks > 1) c->xseq++;                          // peer-memory mode: the plane kernel's last block sums over the ranks itself
    CU(cudaEventRecord(c->ev0, c->stream));
    if (search) {
        if (c->S.n == 0) {
            // an empty slot (more ranks than points): nothing to search
        } else if (c->cells) launch_knn_cells_scan(c, P);
        else switch (c->group ? c->group : group_for(c->S.n)) {
            case 16: launch_knn_scan<16>(c, P); break;
            case 32: launch_knn_scan<32>(c, P); break;
            case 2: launch_knn_scan<2>(c, P); break;
            case 8: launch_knn_scan<8>(c, P); break;
            default: launch_knn_scan<4>(c, P); break;
        }
        CU(cudaEventRecord(c->evm, c->stream));
        if (imu_en) launch_plane<true, true>(c, P, out); else launch_plane<false, true>(c, P, out);
        c->have_neighbors = true;
        c->nbr_epoch = c->map_epoch;
        c->scan_fresh = false;   // the two kernels wrote the neighbour copies / selected for every point of the scan
        c->launches += 2;
        c->last_launches = 2;
        c->last_was_search = true;
    } else {
        if (imu_en) launch_plane<true, false>(c, P, out); else launch_plane<false, false>(c, P, out);
        c->launches += 1;
        c->last_launches = 1;
        c->last_was_search = false;
    }
    CU(cudaEventRecord(c->ev1, c->stream));
    CU(cudaGetLastError());
    c->state_gathered = c->nranks == 1;
#ifndef LI_SIMT_EMUL
    if (c->nranks > 1 && !c->comm_p2p) {
        // the one exchange of the path (SURVEY.md section 8e): sum of [HtH 144 | Htr 12 | res_sq | m | pad 2] over the ranks, on the
        // context's stream, then to wherever the caller wants the block (page-locked host block or its own device buffer)
        NcclApi* N = nccl_api();
        ncclResult_t nr = N->AllReduce(c->d_acc, c->d_red, 160, ncclDouble, ncclSum, c->comm, c->stream);
        if (nr != ncclSuccess) return fail(c, LIINIT_ERR_CUDA, std::string("ncclAllReduce: ") + N->GetErrorString(nr));
        CU(cudaMemcpyAsync(final_out, c->d_red, 160 * sizeof(double), cudaMemcpyDefault, c->stream));
    }
#endif
    return LIINIT_OK;
}

#ifndef LI_SIMT_EMUL
// In-place all-gather of one per-point array (elem bytes per point) over the equal-sized shard slots.
int gather_array(Ctx* c, void* base, size_t elem) {
    NcclApi* N = nccl_api();
    const int cnt = (c->scan_n + c->nranks - 1) / c->nranks;
    const size_t bytes = (size_t)cnt * elem;
    ncclResult_t nr = N->AllGather((const char*)base + (size_t)c->rank * bytes, base, bytes, ncclChar, c->comm, c->stream);
    if (nr != ncclSuccess) return fail(c, LIINIT_ERR_CUDA, std::string("ncclAllGather: ") + N->GetErrorString(nr));
    return LIINIT_OK;
}
#endif

// N > 1: bring the other ranks' per-point results (Nearest_Points, flags, normals, world points) onto this device. Collective:
// every rank makes the same call (liinit_map_incremental and the download hooks do).
int gather_scan_state(Ctx* c) {
    if (c->state_gathered) return LIINIT_OK;
#ifndef LI_SIMT_EMUL
    int r;
    if ((r = gather_array(c, c->d_near_xyz, 5 * sizeof(float4)))) return r;
    if ((r = gather_array(c, c->d_selected, 1))) return r;
    if ((r = gather_array(c, c->d_normvec, sizeof(float4)))) return r;
    if ((r = gather_array(c, c->d_world, sizeof(float4)))) return r;
#endif
    c->state_gathered = true;
    return LIINIT_OK;
}

}  // namespace

struct liinit_ctx {
    Ctx c;
};

extern "C" {

const char* liinit_last_error(const liinit_ctx* h) { return h ? h->c.err.c_str() : g_create_error.c_str(); }

int liinit_create(const liinit_config* cfg, liinit_ctx** out) {
    if (!cfg || !out) {
        g_create_error = "null argument";
        return LIINIT_ERR_INVALID;
    }
    *out = nullptr;
    if (!(cfg->filter_size_map > 0.f) || cfg->max_map_points <= 0 || cfg->max_scan_points <= 0) {
        g_create_error = "filter_size_map, max_map_points and max_scan_points must be positive";
        return LIINIT_ERR_INVALID;
    }
    liinit_ctx* h = new liinit_ctx();
    Ctx* c = &h->c;
    c->cfg = *cfg;
    auto bail = [&](int code) {
        g_create_error = c->err;
        liinit_destroy(h);
        return code;
    };
#define CUC(call)                                                                 \
    do {                                                                          \
        cudaError_t _e = (call);                                                  \
        if (_e != cudaSuccess) {                                                  \
            c->err = std::string(#call) + ": " + cudaGetErrorString(_e);          \
            return bail(LIINIT_ERR_CUDA);                                         \
        }                                                                         \
    } while (0)
    int ndev = 0;
    CUC(cudaGetDeviceCount(&ndev));
    if (cfg->device_id < 0 || cfg->device_id >= ndev) {
        c->err = "device_id out of range (no usable CUDA device; there is no CPU fallback)";
        return bail(LIINIT_ERR_CUDA);
    }
    c->device = cfg->device_id;
    CUC(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    CUC(cudaGetDeviceProperties(&prop, c->device));
    c->num_sms = prop.multiProcessorCount;
    CUC(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    c->stream = c->own_stream;
    CUC(cudaEventCreate(&c->ev0));
    CUC(cudaEventCreate(&c->ev1));
    CUC(cudaEventCreate(&c->evm));

    int bs = cfg->brick_cells_log2 > 0 ? cfg->brick_cells_log2 : 3;
    if (bs < 1 || bs > 4) {
        c->err = "brick_cells_log2 must be in [1,4]";
        return bail(LIINIT_ERR_INVALID);
    }
    int hl = cfg->hash_capacity_log2;
    if (hl <= 0) {
        // ~ one brick per 4 live points worst case for surface maps, load factor <= 0.5
        long long want = (long long)cfg->max_map_points / 2;
        hl = 16;
        while ((1ll << hl) < want && hl < 28) hl++;
    }
    if (hl < 10 || hl > 30) {
        c->err = "hash_capacity_log2 out of range";
        return bail(LIINIT_ERR_INVALID);
    }
    c->hash_slots = 1u << hl;
    // lanes per scan point of the lockstep search: fixed by the caller, or (0) chosen per pass from the frame size (group_for)
    c->group = (cfg->knn_group_lanes == 2 || cfg->knn_group_lanes == 4 || cfg->knn_group_lanes == 8 || cfg->knn_group_lanes == 16 || cfg->knn_group_lanes == 32) ? cfg->knn_group_lanes : 0;
    {
        const char* ge = getenv("LIINIT_KNN_GROUP");   // developer A/B
        if (ge && (atoi(ge) == 2 || atoi(ge) == 4 || atoi(ge) == 8 || atoi(ge) == 16 || atoi(ge) == 32)) c->group = atoi(ge);
    }

    {
        int ki = cfg->knn_index;
        if (ki == 0) {
            // developer A/B switch: run an unmodified caller (tests, bench) against the other index
            const char* e = getenv("LIINIT_KNN_INDEX");
            ki = (e && *e) ? atoi(e) : LIINIT_KNN_DEFAULT;
        }
        if (ki != LIINIT_KNN_BRICKS && ki != LIINIT_KNN_CELLS) {
            c->err = "knn_index must be 0, LIINIT_KNN_BRICKS or LIINIT_KNN_CELLS";
            return bail(LIINIT_ERR_INVALID);
        }
        // the cell directory is defined for 8x8x8-voxel bricks; another brick size keeps the brick search
        c->cells = ki == LIINIT_KNN_CELLS && bs == LI_CELLS_BSHIFT;
        const char* sd = getenv("LIINIT_CELLS_SCHED");
        if (sd && !strcmp(sd, "dynamic")) c->cells_dynamic = true;
        const char* rf = getenv("LIINIT_CELLS_REFRESH");
        if (rf && !strcmp(rf, "thread")) c->cells_refresh_warp = false;
        const char* cs = getenv("LIINIT_CELLS_SEARCH");
        if (cs && atoi(cs) >= 1 && atoi(cs) <= 3) c->cells_search = atoi(cs);
    }
    {
        float cells = cfg->knn_seed_radius_cells > 0.f ? cfg->knn_seed_radius_cells : 2.0f;
        float rho = cells * cfg->filter_size_map;
        c->rho2 = rho * rho;
    }
    MapDev& M = c->M;
    M.mask = c->hash_slots - 1;
    M.ds = cfg->filter_size_map;
    M.bshift = bs;
    // slabs grow geometrically and old slabs are abandoned: 3x live capacity + per-brick minimum slack
    unsigned long long pool = (unsigned long long)cfg->max_map_points * 3ull + (1ull << 20);
    if (pool > 0x7fffff00ull) pool = 0x7fffff00ull;   // ids are int32 pool offsets
    M.pool_cap = pool;
    CUC(cudaMalloc(&M.ent, (size_t)c->hash_slots * sizeof(uint4)));
    CUC(cudaMalloc(&M.brick_slots, (size_t)c->hash_slots * sizeof(int)));
    CUC(cudaMalloc(&M.aux, (size_t)c->hash_slots * sizeof(uint4)));
    CUC(cudaMalloc(&M.pool, (size_t)pool * sizeof(float4)));
    CUC(cudaMalloc(&M.pool_top, sizeof(unsigned long long)));
    M.cocc = nullptr;
    M.cdir = nullptr;
    M.sb_keys = nullptr;
    M.sb_occ = nullptr;
    M.sb_mask = 0;
    if (c->cells) {
        CUC(cudaMalloc(&M.cocc, (size_t)c->hash_slots * sizeof(unsigned long long)));
        CUC(cudaMalloc(&M.cdir, (size_t)c->hash_slots * 64 * sizeof(unsigned short)));
        // one super-brick per brick in the worst case (scattered points): same slot count as the brick hash
        M.sb_mask = c->hash_slots - 1;
        CUC(cudaMalloc(&M.sb_keys, (size_t)c->hash_slots * sizeof(unsigned long long)));
        CUC(cudaMalloc(&M.sb_occ, (size_t)c->hash_slots * sizeof(unsigned long long)));
        CUC(cudaMalloc(&c->d_ticket, sizeof(unsigned)));
    }
    int batch = cfg->max_scan_points > (1 << 20) ? cfg->max_scan_points : (1 << 20);
    c->stage_pts_cap = batch;
    CUC(cudaMalloc(&M.touched_list, (size_t)batch * 2 * sizeof(int)));
    CUC(cudaMalloc(&c->d_counters, sizeof(int) * CNT_COUNT));
    M.counters = c->d_counters;
    CUC(cudaMallocHost(&c->h_counters, sizeof(int) * CNT_COUNT));
    CUC(cudaMallocHost(&c->h_pool_top, sizeof(unsigned long long)));
    *c->h_pool_top = 0;
    c->stage_raw_floats = (size_t)batch * 12;
    CUC(cudaMalloc(&c->d_stage_raw, c->stage_raw_floats * 4));
    CUC(cudaMalloc(&c->d_stage_pts, (size_t)batch * sizeof(float4)));
    CUC(cudaMalloc(&c->d_slot_of, (size_t)batch * sizeof(int)));
    CUC(cudaMalloc(&c->d_vslot_of, (size_t)batch * sizeof(int)));
    CUC(cudaMalloc(&c->d_flag, (size_t)batch * sizeof(int)));
    CUC(cudaMalloc(&c->d_ins, (size_t)batch * sizeof(int)));
    CUC(cudaMalloc(&c->d_q_d2, (size_t)batch * 5 * sizeof(float)));
    {
        int vl = 10;
        while ((1ll << vl) < 2ll * batch) vl++;
        c->V.mask = (1u << vl) - 1;
        CUC(cudaMalloc(&c->V.keys, ((size_t)c->V.mask + 1) * 8));
        CUC(cudaMalloc(&c->V.head, ((size_t)c->V.mask + 1) * 4));
        CUC(cudaMalloc(&c->V.coupled, ((size_t)c->V.mask + 1) * 4));
        CUC(cudaMalloc(&c->V.sum, ((size_t)c->V.mask + 1) * sizeof(int4)));
        CUC(cudaMalloc(&c->V.clist, ((size_t)c->V.mask + 1) * 4));
        CUC(cudaMalloc(&c->d_vg_imin, ((size_t)c->V.mask + 1) * 4));
        CUC(cudaMalloc(&c->d_vg_block, ((size_t)batch / 1024 + 2) * 4));
        CUC(cudaMalloc(&c->d_vg_misc, 8 * 4));
        CUC(cudaMalloc(&c->d_rs_keys, (size_t)batch * 4));
        CUC(cudaMalloc(&c->d_rs_vals, (size_t)batch * 4));
        CUC(cudaMalloc(&c->d_rs_hist, ((size_t)batch / RS_TILE + 2) * 256 * 4));
        CUC(cudaMalloc(&c->d_vg_params, sizeof(VgParams)));
        CUC(cudaMalloc(&c->d_tmin_idx, 8));
        CUC(cudaMalloc(&c->d_poses, 4096 * LI_POSE6D_DOUBLES * sizeof(double)));
    }
    int ns = cfg->max_scan_points + 64;   // (+ slack: equal-sized shard slots of a frame cut over up to 64 ranks)
    CUC(cudaMalloc(&c->d_acc, 160 * sizeof(double)));
    CUC(cudaMalloc(&c->d_red, 160 * sizeof(double)));
    CUC(cudaMalloc(&c->d_body, (size_t)ns * sizeof(float4)));
    CUC(cudaMalloc(&c->d_world, (size_t)ns * sizeof(float4)));
    CUC(cudaMalloc(&c->d_near_ids, (size_t)batch * 5 * sizeof(int)));
    CUC(cudaMalloc(&c->d_near_xyz, (size_t)ns * 5 * sizeof(float4)));
    CUC(cudaMalloc(&c->d_selected, (size_t)ns));
    CUC(cudaMalloc(&c->d_normvec, (size_t)ns * sizeof(float4)));
    c->max_blocks = c->num_sms * 16;
    CUC(cudaMalloc(&c->d_partials, (size_t)c->max_blocks * 96 * sizeof(double)));
    CUC(cudaMalloc(&c->d_done, sizeof(unsigned)));
    CUC(cudaHostAlloc(&c->h_out, 160 * sizeof(double), cudaHostAllocMapped));
    CUC(cudaHostGetDevicePointer((void**)&c->h_out_dev, c->h_out, 0));
    CUC(cudaMemsetAsync(c->d_done, 0, sizeof(unsigned), c->stream));
    CUC(cudaMemsetAsync(c->d_counters, 0, sizeof(int) * CNT_COUNT, c->stream));
    CUC(cudaMemsetAsync(M.pool_top, 0, sizeof(unsigned long long), c->stream));
    k_map_clear<<<nblk(c->hash_slots, 256), 256, 0, c->stream>>>(M.ent, M.aux, c->hash_slots);
    c->launches++;
    if (c->cells) {
        k_sb_clear<<<nblk(c->hash_slots, 256), 256, 0, c->stream>>>(M);
        c->launches++;
    }
    CUC(cudaGetLastError());
    CUC(cudaStreamSynchronize(c->stream));
    c->S.body = c->d_body;
    c->S.world = c->d_world;
    c->S.near_ids = c->d_near_ids;
    c->S.near_xyz = c->d_near_xyz;
    c->S.selected = c->d_selected;
    c->S.normvec = c->d_normvec;
    c->S.n = 0;
#undef CUC
    *out = h;
    return LIINIT_OK;
}

int liinit_destroy(liinit_ctx* h) {
    if (!h) return LIINIT_OK;
    Ctx* c = &h->c;
    cudaSetDevice(c->device);
    if (c->own_stream) cudaStreamSynchronize(c->own_stream);
    cudaFree(c->M.ent); cudaFree(c->M.brick_slots); cudaFree(c->M.aux); cudaFree(c->M.pool); cudaFree(c->M.pool_top); cudaFree(c->M.touched_list); cudaFree(c->M.cocc); cudaFree(c->M.cdir); cudaFree(c->M.sb_keys); cudaFree(c->M.sb_occ); cudaFree(c->d_ticket);
    cudaFree(c->d_counters); cudaFreeHost(c->h_counters); cudaFreeHost(c->h_pool_top); cudaFree(c->d_stage_raw); cudaFree(c->d_stage_pts);
    cudaFree(c->d_slot_of); cudaFree(c->d_vslot_of); cudaFree(c->d_flag); cudaFree(c->d_ins); cudaFree(c->V.keys); cudaFree(c->V.head); cudaFree(c->V.coupled); cudaFree(c->V.sum); cudaFree(c->V.clist); cudaFree(c->d_vg_imin); cudaFree(c->d_vg_block); cudaFree(c->d_vg_misc); cudaFree(c->d_rs_keys); cudaFree(c->d_rs_vals); cudaFree(c->d_rs_hist); cudaFree(c->d_vg_params); cudaFree(c->d_tmin_idx); cudaFree(c->d_poses);
    cudaFree(c->d_body); cudaFree(c->d_world); cudaFree(c->d_near_ids); cudaFree(c->d_near_xyz); cudaFree(c->d_selected); cudaFree(c->d_normvec);
    cudaFree(c->d_acc); cudaFree(c->d_red);
#ifndef LI_SIMT_EMUL
    for (int r = 0; r < LI_MAX_RANKS; r++)
        if (c->peer_map[r]) cudaIpcCloseMemHandle(c->peer_map[r]);
    cudaFree(c->d_xtab);
    cudaFree(c->d_xbuf);
    if (c->comm) { NcclApi* N = nccl_api(); if (N) N->CommDestroy(c->comm); c->comm = nullptr; }
#endif
    cudaFree(c->d_partials); cudaFree(c->d_done); cudaFreeHost(c->h_out); cudaFree(c->d_q_d2);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->evm) cudaEventDestroy(c->evm);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete h;
    return LIINIT_OK;
}

int liinit_set_stream(liinit_ctx* h, void* cuda_stream) {
    if (!h) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    c->stream = cuda_stream ? (cudaStream_t)cuda_stream : c->own_stream;
    return LIINIT_OK;
}

int liinit_map_build(liinit_ctx* h, const float* xyz, int stride, int n) {
    if (!h || (!xyz && n > 0) || n < 0) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    if (n > c->cfg.max_map_points) return fail(c, LIINIT_ERR_CAPACITY, "n exceeds max_map_points");
    c->map_epoch++;
    c->map_version++;
    // KD_TREE::Build replaces the tree (ikd_Tree.cpp:337-339)
    CU(cudaMemsetAsync(c->d_counters, 0, sizeof(int) * CNT_COUNT, c->stream));
    CU(cudaMemsetAsync(c->M.pool_top, 0, sizeof(unsigned long long), c->stream));
    k_map_clear<<<nblk(c->hash_slots, 256), 256, 0, c->stream>>>(c->M.ent, c->M.aux, c->hash_slots);
    c->launches++;
    if (c->cells) {
        k_sb_clear<<<nblk(c->hash_slots, 256), 256, 0, c->stream>>>(c->M);
        c->launches++;
    }
    // (the retained Nearest_Points are copies: a reuse pass / map_incremental after a map change works on them as in the reference)
    for (long long off = 0; off < n; off += c->stage_pts_cap) {
        int m = (int)((n - off < c->stage_pts_cap) ? (n - off) : c->stage_pts_cap);
        int r = stage_points(c, xyz + (size_t)off * stride, stride, m);
        if (r) return r;
        r = plain_insert(c, c->d_stage_pts, m, nullptr, 0);
        if (r) return r;
        // the staging buffers are reused by the next chunk
        CU(cudaStreamSynchronize(c->stream));
    }
    int r = fetch_counters(c);
    if (r) return r;
    return check_map_err(c);
}

}  // extern "C"

namespace {
// Slabs only ever grow from the bump allocator and a brick emptied by deletes keeps its slab and its hash slot: a sliding local map
// (Add_Points ahead, Delete_Point_Boxes behind) would run the pool dry although few points are alive. Compaction = flatten the live
// points, clear hash + pool, re-insert them (the Build path): every brick gets one tight slab, empty bricks disappear.
int compact_map(Ctx* c) {
    c->map_epoch++;
    c->map_version++;
    int r = fetch_counters(c);
    if (r) return r;
    const int live = c->h_counters[CNT_LIVE];
    DevBuf<float4> btmp;
    DevBuf<int> bn;
    float4* d_tmp = nullptr;
    int* d_n = nullptr;
    if (live > 0) {
        CU(btmp.alloc((size_t)live));
        CU(bn.alloc(1));
        d_tmp = btmp.p;
        d_n = bn.p;
        CU(cudaMemsetAsync(d_n, 0, sizeof(int), c->stream));
        k_map_flatten4<<<nblk((long long)c->h_counters[CNT_BRICKS] * 32, 256), 256, 0, c->stream>>>(c->M, c->hash_slots, d_tmp, live, d_n);
        c->launches++;
    }
    CU(cudaMemsetAsync(c->d_counters, 0, sizeof(int) * CNT_COUNT, c->stream));
    CU(cudaMemsetAsync(c->M.pool_top, 0, sizeof(unsigned long long), c->stream));
    k_map_clear<<<nblk(c->hash_slots, 256), 256, 0, c->stream>>>(c->M.ent, c->M.aux, c->hash_slots);
    c->launches++;
    if (c->cells) {
        k_sb_clear<<<nblk(c->hash_slots, 256), 256, 0, c->stream>>>(c->M);
        c->launches++;
    }
    r = LIINIT_OK;
    for (long long off = 0; off < live && r == LIINIT_OK; off += c->stage_pts_cap) {
        const int m = (int)((live - off < c->stage_pts_cap) ? (live - off) : c->stage_pts_cap);
        r = plain_insert(c, d_tmp + off, m, nullptr, 0);
    }
    if (r == LIINIT_OK) r = fetch_counters(c);   // (synchronises: the scratch may go)
    else cudaStreamSynchronize(c->stream);
    if (r) return r;
    return check_map_err(c);
}

// Before an update of up to `incoming` points: compact when the allocator is in its last quarter and at least half of what it
// handed out is dead (abandoned slabs, deleted points).
int maybe_compact(Ctx* c, long long incoming) {
    const unsigned long long top = *c->h_pool_top, cap = c->M.pool_cap;
    const long long live = c->h_counters[CNT_LIVE];
    if (top + (unsigned long long)(3 * incoming) + (1ull << 16) > cap - cap / 4 && (unsigned long long)(2 * live) < top) return compact_map(c);
    return LIINIT_OK;
}
}  // namespace

extern "C" {

int liinit_map_compact(liinit_ctx* h) {
    if (!h) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    return compact_map(c);
}

int liinit_map_add_points(liinit_ctx* h, const float* xyz, int stride, int n, int downsample_on, int* added) {
    if (!h || (!xyz && n > 0) || n < 0) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    c->map_epoch++;
    c->map_version++;
    {
        int r = maybe_compact(c, n);
        if (r) return r;
    }
    int total = 0;
    for (long long off = 0; off < n; off += c->stage_pts_cap) {
        int m = (int)((n - off < c->stage_pts_cap) ? (n - off) : c->stage_pts_cap);
        int r = stage_points(c, xyz + (size_t)off * stride, stride, m);
        if (r) return r;
        r = downsample_on ? downsample_insert(c, c->d_stage_pts, m, nullptr, 0) : plain_insert(c, c->d_stage_pts, m, nullptr, 0);
        if (r) return r;
        r = fetch_counters(c);
        if (r) return r;
        r = check_map_err(c);
        if (r) return r;
        total += downsample_on ? c->h_counters[CNT_CHANGED] : m;
    }
    if (added) *added = total;
    return LIINIT_OK;
}

int liinit_map_delete_boxes(liinit_ctx* h, const float* boxes, int nbox, int* deleted) {
    if (!h || (!boxes && nbox > 0) || nbox < 0) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    if (deleted) *deleted = 0;
    if (nbox == 0) return LIINIT_OK;
    c->map_epoch++;
    c->map_version++;
    if ((size_t)nbox * 6 > c->stage_raw_floats) return fail(c, LIINIT_ERR_CAPACITY, "too many boxes");
    CU(cudaMemcpyAsync(c->d_stage_raw, boxes, (size_t)nbox * 6 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemsetAsync(c->d_vg_misc + 6, 0, sizeof(int), c->stream));
    {   // bricks created so far (the counters are fetched at the end of every map update)
        int r = fetch_counters(c);
        if (r) return r;
    }
    if (c->h_counters[CNT_BRICKS] <= 0) return LIINIT_OK;
    k_map_delete_boxes<<<nblk((long long)c->h_counters[CNT_BRICKS] * 32, 256), 256, 0, c->stream>>>(c->M, c->hash_slots, c->d_stage_raw, nbox,
                                                                                          c->d_vg_misc + 6);
    c->launches++;
    if (c->cells) {
        if (c->cells_refresh_warp) k_cells_refresh_all_warp<<<c->num_sms * 16, 128, 0, c->stream>>>(c->M, c->hash_slots);
        else k_cells_refresh_all<<<nblk(c->hash_slots, 128), 128, 0, c->stream>>>(c->M, c->hash_slots);
        c->launches++;
    }
    CU(cudaGetLastError());
    int cnt = 0;
    CU(cudaMemcpyAsync(&cnt, c->d_vg_misc + 6, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (deleted) *deleted = cnt;
    return LIINIT_OK;
}

int liinit_map_validnum(liinit_ctx* h, int* n) {
    if (!h || !n) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    int r = fetch_counters(c);
    if (r) return r;
    *n = c->h_counters[CNT_LIVE];
    return LIINIT_OK;
}

int liinit_map_size(liinit_ctx* h, int* n) { return liinit_map_validnum(h, n); }

int liinit_map_stats(liinit_ctx* h, int* bricks, int* hash_slots, long long* pool_used, long long* pool_cap) {
    if (!h) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    int r = fetch_counters(c);
    if (r) return r;
    unsigned long long top = 0;
    CU(cudaMemcpyAsync(&top, c->M.pool_top, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (bricks) *bricks = c->h_counters[CNT_BRICKS];
    if (hash_slots) *hash_slots = (int)c->hash_slots;
    if (pool_used) *pool_used = (long long)top;
    if (pool_cap) *pool_cap = (long long)c->M.pool_cap;
    return LIINIT_OK;
}

int liinit_map_download(liinit_ctx* h, float* xyz, int cap, int* n) {
    if (!h || !n || cap < 0) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    DevBuf<float> out;
    DevBuf<int> dn;
    CU(out.alloc((size_t)(cap > 0 ? cap : 1) * 3));
    CU(dn.alloc(1));
    float* d_out = out.p;
    int* d_n = dn.p;
    CU(cudaMemsetAsync(d_n, 0, 4, c->stream));
    {
        int r = fetch_counters(c);
        if (r) return r;
    }
    if (c->h_counters[CNT_BRICKS] > 0)
        k_map_flatten<<<nblk((long long)c->h_counters[CNT_BRICKS] * 32, 256), 256, 0, c->stream>>>(c->M, c->hash_slots, d_out, cap, d_n);
    c->launches++;
    CU(cudaGetLastError());
    int cnt = 0;
    CU(cudaMemcpyAsync(&cnt, d_n, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    int m = cnt < cap ? cnt : cap;
    if (m > 0 && xyz) CU(cudaMemcpy(xyz, d_out, (size_t)m * 12, cudaMemcpyDeviceToHost));
    *n = cnt;
    return LIINIT_OK;
}

int liinit_map_nearest_search(liinit_ctx* h, const float* q, int stride, int n, double max_dist, float* out_xyz, float* out_d2,
                              int* out_cnt) {
    if (!h || !q || n < 0) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    if (max_dist != 5.0) return fail(c, LIINIT_ERR_INVALID, "only max_dist = 5 (laserMapping.cpp:980) is supported");
    CU(cudaSetDevice(c->device));
    std::vector<int> ids((size_t)5 * (n > 0 ? n : 1));
    for (long long off = 0; off < n; off += c->stage_pts_cap) {
        int m = (int)((n - off < c->stage_pts_cap) ? (n - off) : c->stage_pts_cap);
        int r = stage_points(c, q + (size_t)off * stride, stride, m);
        if (r) return r;
        DevBuf<int> bids;
        DevBuf<float> bxyz;
        CU(bids.alloc((size_t)m * 5));
        CU(bxyz.alloc((size_t)m * 15));
        int* d_ids = bids.p;
        float* d_xyz = bxyz.p;
        if (c->cells) {
            const int gq = nblk(m, LI_CELLS_THREADS);
            if (c->cells_search == 1) k_knn_cells_queries<1><<<gq, LI_CELLS_THREADS, 0, c->stream>>>(c->M, c->d_stage_pts, m, d_ids, c->d_q_d2, c->rho2);
            else if (c->cells_search == 2) k_knn_cells_queries<2><<<gq, LI_CELLS_THREADS, 0, c->stream>>>(c->M, c->d_stage_pts, m, d_ids, c->d_q_d2, c->rho2);
            else k_knn_cells_queries<3><<<gq, LI_CELLS_THREADS, 0, c->stream>>>(c->M, c->d_stage_pts, m, d_ids, c->d_q_d2, c->rho2);
        } else {
            int grid = nblk((long long)m * 8, 256);
            if (grid > c->max_blocks) grid = c->max_blocks;
            k_knn_queries<8><<<grid, 256, 0, c->stream>>>(c->M, c->d_stage_pts, m, d_ids, c->d_q_d2, c->rho2);
        }
        k_gather_xyz<<<nblk((long long)m * 5, 256), 256, 0, c->stream>>>(c->M.pool, d_ids, (long long)m * 5, d_xyz);
        c->launches += 2;
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(ids.data() + (size_t)off * 5, d_ids, (size_t)m * 5 * 4, cudaMemcpyDeviceToHost, c->stream));
        if (out_xyz) CU(cudaMemcpyAsync(out_xyz + (size_t)off * 15, d_xyz, (size_t)m * 15 * 4, cudaMemcpyDeviceToHost, c->stream));
        if (out_d2) CU(cudaMemcpyAsync(out_d2 + (size_t)off * 5, c->d_q_d2, (size_t)m * 5 * 4, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
    }
    for (int i = 0; i < n; i++) {
        int cnt = 0;
        for (int k = 0; k < 5; k++)
            if (ids[(size_t)i * 5 + k] >= 0) cnt++;
        if (out_cnt) out_cnt[i] = cnt;
        // PointType_CMP tie order (ikd_Tree.h:57-60)
        if (out_xyz && out_d2) {
            for (int pass = 0; pass < 4; pass++)
                for (int k = 0; k + 1 < cnt; k++) {
                    size_t a = (size_t)i * 5 + k, b = a + 1;
                    if (std::fabs(out_d2[a] - out_d2[b]) < 1e-10f && out_xyz[3 * b] < out_xyz[3 * a]) {
                        for (int t = 0; t < 3; t++) std::swap(out_xyz[3 * a + t], out_xyz[3 * b + t]);
                        std::swap(out_d2[a], out_d2[b]);
                    }
                }
        }
    }
    return LIINIT_OK;
}

}  // extern "C"

namespace {
// The reference compares the float d2 with the double max_dist (ikd_Tree.cpp:842): d2 <= max_dist <=> d2 <= the largest float not above
// max_dist. (float)max_dist rounds to nearest and would admit points the reference rejects whenever max_dist is not a float.
float float_at_most(double v) {
    float f = (float)v;
    if ((double)f > v) f = std::nextafter(f, -INFINITY);
    return f;
}

int knn_args_check(Ctx* c, int stride, int n, int k, double max_dist) {
    if (k < 1 || k > LIINIT_KNN_MAX_K) return fail(c, LIINIT_ERR_INVALID, "k must be in 1.." + std::to_string(LIINIT_KNN_MAX_K));
    if (!(max_dist >= 0.0)) return fail(c, LIINIT_ERR_INVALID, "max_dist must be >= 0 or +INFINITY (not NaN)");
    if (n < 0) return fail(c, LIINIT_ERR_INVALID, "n must be >= 0");
    if (stride != 3 && stride != 4 && stride != 12) return fail(c, LIINIT_ERR_INVALID, "stride_floats must be 3, 4 or 12");
    return LIINIT_OK;
}

// The search itself, queued on the context's stream: queries and outputs are device memory.
int knn_general(Ctx* c, const float* d_q, int stride, int n, int k, double max_dist, float* d_xyz, float* d_d2, int* d_cnt) {
    if (n == 0) return LIINIT_OK;
    if (!c->knn_occ.p) CU(c->knn_occ.alloc(c->hash_slots));
    if (!c->knn_occ_valid || c->knn_occ_version != c->map_version) {
        k_knn_occ_build<<<c->num_sms * 4, 256, 0, c->stream>>>(c->M, c->knn_occ.p);
        c->launches++;
        c->knn_occ_version = c->map_version;
        c->knn_occ_valid = true;
    }
    const int wpb = LI_KNN_GEN_THREADS / 32;
    long long grid = ((long long)n + wpb - 1) / wpb;
    if (grid > c->max_blocks) grid = c->max_blocks;
    k_knn_general<<<(int)grid, LI_KNN_GEN_THREADS, 0, c->stream>>>(c->M, c->knn_occ.p, d_q, stride, n, k, float_at_most(max_dist), c->rho2, d_xyz, d_d2,
                                                                   d_cnt);
    c->launches++;
    CU(cudaGetLastError());
    return LIINIT_OK;
}
}  // namespace

extern "C" {

int liinit_map_knn_search_device(liinit_ctx* h, const float* d_q, int stride, int n, int k, double max_dist, float* d_out_xyz, float* d_out_d2,
                                 int* d_out_cnt) {
    if (!h) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    if ((n > 0 && (!d_q || !d_out_xyz || !d_out_d2 || !d_out_cnt))) return fail(c, LIINIT_ERR_INVALID, "null pointer");
    int r = knn_args_check(c, stride, n, k, max_dist);
    if (r) return r;
    CU(cudaSetDevice(c->device));
    return knn_general(c, d_q, stride, n, k, max_dist, d_out_xyz, d_out_d2, d_out_cnt);
}

int liinit_map_knn_search(liinit_ctx* h, const float* q, int stride, int n, int k, double max_dist, float* out_xyz, float* out_d2, int* out_cnt) {
    if (!h) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    if (n > 0 && (!q || !out_xyz || !out_d2 || !out_cnt)) return fail(c, LIINIT_ERR_INVALID, "null pointer");
    int r = knn_args_check(c, stride, n, k, max_dist);
    if (r) return r;
    CU(cudaSetDevice(c->device));
    if (n == 0) return LIINIT_OK;
    const int chunk = n < c->stage_pts_cap ? n : c->stage_pts_cap;
    DevBuf<float> bxyz, bd2;
    DevBuf<int> bcnt;
    CU(bxyz.alloc((size_t)chunk * k * 3));
    CU(bd2.alloc((size_t)chunk * k));
    CU(bcnt.alloc((size_t)chunk));
    for (long long off = 0; off < n; off += c->stage_pts_cap) {
        const int m = (int)((n - off < c->stage_pts_cap) ? (n - off) : c->stage_pts_cap);
        r = stage_points(c, q + (size_t)off * stride, stride, m);
        if (r) return r;
        r = knn_general(c, reinterpret_cast<const float*>(c->d_stage_pts), 4, m, k, max_dist, bxyz.p, bd2.p, bcnt.p);
        if (r) return r;
        CU(cudaMemcpyAsync(out_xyz + (size_t)off * k * 3, bxyz.p, (size_t)m * k * 3 * 4, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaMemcpyAsync(out_d2 + (size_t)off * k, bd2.p, (size_t)m * k * 4, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaMemcpyAsync(out_cnt + off, bcnt.p, (size_t)m * 4, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));   // the staging buffer is reused by the next chunk
    }
    return LIINIT_OK;
}

int liinit_scan_upload(liinit_ctx* h, const float* body, int stride, int n) {
    if (!h || !body || n <= 0) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    if (n > c->cfg.max_scan_points) return fail(c, LIINIT_ERR_CAPACITY, "n exceeds max_scan_points");
    c->attached = nullptr;
    c->attached_slot_done = false;
    if (stride == 4) {
        CU(cudaMemcpyAsync(c->d_body, body, (size_t)n * 16, cudaMemcpyHostToDevice, c->stream));
    } else if (stride == 3 || stride == 12) {
        size_t nf = (size_t)n * stride;
        if (nf > c->stage_raw_floats) return fail(c, LIINIT_ERR_CAPACITY, "scan exceeds staging capacity");
        CU(cudaMemcpyAsync(c->d_stage_raw, body, nf * 4, cudaMemcpyHostToDevice, c->stream));
        k_repack<<<nblk(n, 256), 256, 0, c->stream>>>(c->d_stage_raw, stride, n, c->d_body);
        c->launches++;
    } else {
        return fail(c, LIINIT_ERR_INVALID, "stride_floats must be 3, 4 or 12");
    }
    // new scan: no neighbours, nothing selected (Nearest_Points / point_selected_surf start over at iteration 0)
    set_scan(c, n);
    CU(cudaGetLastError());
    return LIINIT_OK;
}

int liinit_scan_attach_host(liinit_ctx* h, const float* pinned_body, int stride, int n) {
    if (!h || !pinned_body || n <= 0) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    if (n > c->cfg.max_scan_points) return fail(c, LIINIT_ERR_CAPACITY, "n exceeds max_scan_points");
    if (stride != 3 && stride != 4 && stride != 12) return fail(c, LIINIT_ERR_INVALID, "stride_floats must be 3, 4 or 12");
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, pinned_body) != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer) {
        cudaGetLastError();
        return fail(c, LIINIT_ERR_INVALID, "scan_attach_host needs page-locked, device-mapped host memory (cudaHostAlloc / cudaHostRegister)");
    }
    c->attached = (const float*)at.devicePointer;
    c->attached_stride = stride;
    c->attached_slot_done = false;
    set_scan(c, n);   // (N > 1: the search kernel reads this rank's slot in place; the rest is copied when map_incremental / a download needs it)
    return LIINIT_OK;
}

int liinit_raw_upload(liinit_ctx* h, const float* pts, int stride, int time_index, int n) {
    if (!h || !pts || n <= 0) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    if (stride < 3 || time_index >= stride || (time_index >= 0 && time_index < 3)) return fail(c, LIINIT_ERR_INVALID, "bad stride / time_index");
    if (n > c->stage_pts_cap || (size_t)n * stride > c->stage_raw_floats) return fail(c, LIINIT_ERR_CAPACITY, "raw cloud exceeds staging capacity");
    CU(cudaMemcpyAsync(c->d_stage_raw, pts, (size_t)n * stride * 4, cudaMemcpyHostToDevice, c->stream));
    k_repack_t<<<nblk(n, 256), 256, 0, c->stream>>>(c->d_stage_raw, stride, time_index, n, c->d_stage_pts);
    c->launches++;
    c->raw_n = n;
    CU(cudaGetLastError());
    return LIINIT_OK;
}

static int raw_time_range(Ctx* c) {
    const int neg = (int)0xff800000 ^ 0x7fffffff;   // ordered-int image of -inf
    const unsigned long long big = ~0ull;
    CU(cudaMemcpyAsync(c->d_vg_misc + 5, &neg, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->d_tmin_idx, &big, 8, cudaMemcpyHostToDevice, c->stream));
    k_time_range<<<nblk(c->raw_n, 256), 256, 0, c->stream>>>(c->d_stage_pts, c->raw_n, c->d_tmin_idx, c->d_vg_misc + 5);
    c->launches++;
    return LIINIT_OK;
}

int liinit_raw_undistort_cv(liinit_ctx* h, const double omega[3], const double rot_end[9], const double vel_end[3]) {
    if (!h || !omega || !rot_end || !vel_end) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    if (c->raw_n <= 0) return fail(c, LIINIT_ERR_INVALID, "no raw cloud staged (liinit_raw_upload)");
    int r = raw_time_range(c);
    if (r) return r;
    CvParams P;
    for (int a = 0; a < 3; a++) {
        P.omega[a] = omega[a];
        P.vb[a] = rot_end[a] * vel_end[0] + rot_end[3 + a] * vel_end[1] + rot_end[6 + a] * vel_end[2];   // rot_end^T vel_end
    }
    k_undistort_cv<<<nblk(c->raw_n, 256), 256, 0, c->stream>>>(c->d_stage_pts, c->raw_n, P, c->d_vg_misc + 5, c->d_tmin_idx);
    c->launches++;
    CU(cudaGetLastError());
    return LIINIT_OK;
}

int liinit_raw_undistort_imu(liinit_ctx* h, const double* poses, int npose, const double rot_end[9], const double pos_end[3],
                             const double R_LI[9], const double T_LI[3]) {
    if (!h || !poses || npose < 2 || !rot_end || !pos_end || !R_LI || !T_LI) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    if (c->raw_n <= 0) return fail(c, LIINIT_ERR_INVALID, "no raw cloud staged (liinit_raw_upload)");
    if (npose > 4096) return fail(c, LIINIT_ERR_CAPACITY, "IMU pose table too long");
    CU(cudaMemcpyAsync(c->d_poses, poses, (size_t)npose * LI_POSE6D_DOUBLES * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    PoseD S;
    fill_pose(S, rot_end, pos_end, R_LI, T_LI);
    k_undistort_imu<<<nblk(c->raw_n, 256), 256, 0, c->stream>>>(c->d_stage_pts, c->raw_n, c->d_poses, npose, S);
    c->launches++;
    CU(cudaGetLastError());
    return LIINIT_OK;
}

int liinit_raw_download(liinit_ctx* h, float* xyz, int cap, int* n) {
    if (!h || !n) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    *n = c->raw_n;
    int m = c->raw_n < cap ? c->raw_n : cap;
    if (m > 0 && xyz) {
        std::vector<float4> b(m);
        CU(cudaStreamSynchronize(c->stream));
        CU(cudaMemcpy(b.data(), c->d_stage_pts, (size_t)m * 16, cudaMemcpyDeviceToHost));
        for (int i = 0; i < m; i++) {
            xyz[3 * (size_t)i] = b[i].x; xyz[3 * (size_t)i + 1] = b[i].y; xyz[3 * (size_t)i + 2] = b[i].z;
        }
    }
    return LIINIT_OK;
}

int liinit_raw_downsample(liinit_ctx* h, float leaf_size, int* n_down) {
    if (!h || !(leaf_size > 0.f)) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    const int n = c->raw_n;
    if (n <= 0) return fail(c, LIINIT_ERR_INVALID, "no raw cloud staged (liinit_raw_upload)");
    const int inf_pos = 0x7f800000, inf_neg = (int)0xff800000 ^ 0x7fffffff;   // ordered-int images of +inf / -inf
    const int init[8] = {inf_pos, inf_pos, inf_pos, inf_neg, inf_neg, inf_neg, 0, 0};
    CU(cudaMemcpyAsync(c->d_vg_misc, init, sizeof(init), cudaMemcpyHostToDevice, c->stream));
    const int nb = nblk(n, 1024);
    VoxTmp V = sized_vox(c, n);
    k_vg_clear<<<nblk((long long)V.mask + 1, 256), 256, 0, c->stream>>>(V, c->d_vg_imin);
    k_vg_minmax<<<nblk(n, 256), 256, 0, c->stream>>>(c->d_stage_pts, n, c->d_vg_misc);
    k_vg_params<<<1, 32, 0, c->stream>>>(c->d_vg_misc, leaf_size, c->d_vg_params);
    k_vg_link<<<nblk(n, 256), 256, 0, c->stream>>>(c->d_stage_pts, n, c->d_vg_params, V, c->d_vg_imin, c->d_vslot_of, c->d_slot_of,
                                                     c->d_vg_misc + 7);
    // one (leaf index, first point) pair per leaf, sorted by leaf index: PCL's output order
    unsigned* k0 = reinterpret_cast<unsigned*>(c->d_flag);
    unsigned* v0 = reinterpret_cast<unsigned*>(c->d_ins);
    unsigned* k1 = c->d_rs_keys;
    unsigned* v1 = c->d_rs_vals;
    k_vg_collect<<<nblk((long long)V.mask + 1, 256), 256, 0, c->stream>>>(V, c->d_vg_imin, k0, v0, c->d_vg_misc + 6);
    {
        // the number of leaves is only known on the device: sort with the worst-case tile count, the kernels read the real n
        const int ntiles = nblk(n, RS_TILE);
        for (int pass = 0; pass < 4; pass++) {
            k_rs_hist_dev<<<nblk(ntiles, 4), 128, 0, c->stream>>>(k0, c->d_vg_misc + 6, 8 * pass, ntiles, c->d_rs_hist);
            k_rs_scan<<<1, 1024, 0, c->stream>>>(256 * ntiles, c->d_rs_hist);
            k_rs_scatter_dev<<<nblk(ntiles, 4), 128, 0, c->stream>>>(k0, v0, c->d_vg_misc + 6, 8 * pass, ntiles, c->d_rs_hist, k1, v1);
            unsigned* t = k0; k0 = k1; k1 = t;
            t = v0; v0 = v1; v1 = t;
        }
    }
    (void)nb;
    k_vg_centroid_sorted<<<nblk(n, 256), 256, 0, c->stream>>>(c->d_stage_pts, v0, c->d_vg_misc + 6, c->d_slot_of, V, c->d_vslot_of, c->d_body,
                                                               c->cfg.max_scan_points, c->d_vg_misc + 7);
    c->launches += 12;
    c->launches += 7;
    CU(cudaGetLastError());
    int res[8];
    VgParams P;
    CU(cudaMemcpyAsync(res, c->d_vg_misc, sizeof(res), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(&P, c->d_vg_params, sizeof(P), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (P.overflow) return fail(c, LIINIT_ERR_INVALID, "voxel grid: leaf size too small for the cloud extent (index overflow) or no finite point");
    if (res[7] & 1) return fail(c, LIINIT_ERR_CAPACITY, "voxel grid: leaf hash full");
    if (res[7] & 2) return fail(c, LIINIT_ERR_CAPACITY, "voxel grid: more leaves than max_scan_points");
    const int m = res[6];
    if (m <= 0) return fail(c, LIINIT_ERR_INVALID, "voxel grid: no output points");
    set_scan(c, m);
    c->attached = nullptr;
    if (n_down) *n_down = m;
    return LIINIT_OK;
}

int liinit_scan_upload_raw(liinit_ctx* h, const float* xyz, int stride, int n, float leaf_size, int* n_down) {
    int r = liinit_raw_upload(h, xyz, stride, -1, n);
    if (r) return r;
    return liinit_raw_downsample(h, leaf_size, n_down);
}

int liinit_scan_download_body(liinit_ctx* h, float* xyz, int cap, int* n) {
    if (!h || !n) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    *n = c->scan_n;
    int m = c->scan_n < cap ? c->scan_n : cap;
    if (m > 0 && xyz) {
        materialize_scan(c);
        std::vector<float4> b(m);
        CU(cudaStreamSynchronize(c->stream));
        CU(cudaMemcpy(b.data(), c->d_body, (size_t)m * 16, cudaMemcpyDeviceToHost));
        for (int i = 0; i < m; i++) {
            xyz[3 * (size_t)i] = b[i].x; xyz[3 * (size_t)i + 1] = b[i].y; xyz[3 * (size_t)i + 2] = b[i].z;
        }
    }
    return LIINIT_OK;
}

int liinit_icp_iterate_device(liinit_ctx* h, const double* R, const double* p, const double* RLI, const double* TLI, int imu_en,
                              int search, double* d_out160) {
    if (!h || !R || !p || !RLI || !TLI || !d_out160) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    return run_pass(c, R, p, RLI, TLI, imu_en, search, d_out160);
}

int liinit_icp_iterate(liinit_ctx* h, const double* R, const double* p, const double* RLI, const double* TLI, int imu_en,
                       int search, double* HtH, double* Htr, int* m, double* res_sq) {
    if (!h || !R || !p || !RLI || !TLI || !HtH || !Htr || !m) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    int r = run_pass(c, R, p, RLI, TLI, imu_en, search, c->h_out_dev);
    if (r) return r;
    CU(cudaStreamSynchronize(c->stream));
    memcpy(HtH, c->h_out, 144 * sizeof(double));
    memcpy(Htr, c->h_out + 144, 12 * sizeof(double));
    if (res_sq) *res_sq = c->h_out[156];
    *m = (int)llround(c->h_out[157]);
    return LIINIT_OK;
}

int liinit_scan_download_state(liinit_ctx* h, float* world_xyz, float* near_xyz, int* near_cnt, unsigned char* selected,
                               float* normvec) {
    if (!h) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    int n = c->scan_n;
    if (n <= 0) return fail(c, LIINIT_ERR_INVALID, "no scan uploaded");
    {
        int r = init_scan_state(c);
        if (r) return r;
        r = gather_scan_state(c);
        if (r) return r;
    }
    CU(cudaStreamSynchronize(c->stream));
    if (world_xyz) {
        std::vector<float4> w(n);
        CU(cudaMemcpy(w.data(), c->d_world, (size_t)n * 16, cudaMemcpyDeviceToHost));
        for (int i = 0; i < n; i++) {
            world_xyz[3 * (size_t)i] = w[i].x; world_xyz[3 * (size_t)i + 1] = w[i].y; world_xyz[3 * (size_t)i + 2] = w[i].z;
        }
    }
    if (near_xyz || near_cnt) {   // Nearest_Points: the device keeps them as point copies (ScanDev::near_xyz, w = 1 found / 0 missing)
        std::vector<float4> nb((size_t)n * 5);
        CU(cudaMemcpy(nb.data(), c->d_near_xyz, (size_t)n * 5 * sizeof(float4), cudaMemcpyDeviceToHost));
        for (int i = 0; i < n; i++) {
            int cnt = 0;
            for (int k = 0; k < 5; k++) {
                const float4& e = nb[(size_t)i * 5 + k];
                const bool ok = e.w != 0.f;
                if (ok) cnt++;
                if (near_xyz) {
                    float* o = near_xyz + 3 * ((size_t)i * 5 + k);
                    o[0] = ok ? e.x : 0.f; o[1] = ok ? e.y : 0.f; o[2] = ok ? e.z : 0.f;
                }
            }
            if (near_cnt) near_cnt[i] = cnt;
        }
    }
    if (selected) CU(cudaMemcpy(selected, c->d_selected, (size_t)n, cudaMemcpyDeviceToHost));
    if (normvec) CU(cudaMemcpy(normvec, c->d_normvec, (size_t)n * 16, cudaMemcpyDeviceToHost));
    return LIINIT_OK;
}

int liinit_scan_download_effect(liinit_ctx* h, float* ori_xyz, float* normvec, int cap, int* m) {
    if (!h || !m) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    int n = c->scan_n;
    if (n <= 0) return fail(c, LIINIT_ERR_INVALID, "no scan uploaded");
    materialize_scan(c);
    {
        int r = init_scan_state(c);
        if (r) return r;
        r = gather_scan_state(c);
        if (r) return r;
    }
    CU(cudaStreamSynchronize(c->stream));
    std::vector<unsigned char> sel(n);
    std::vector<float4> nv(n), body(n);
    CU(cudaMemcpy(sel.data(), c->d_selected, (size_t)n, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(nv.data(), c->d_normvec, (size_t)n * 16, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(body.data(), c->d_body, (size_t)n * 16, cudaMemcpyDeviceToHost));
    int k = 0;
    for (int i = 0; i < n; i++) {   // order-preserving compaction (laserMapping.cpp:1013-1020)
        if (!sel[i]) continue;
        if (k < cap) {
            if (ori_xyz) {
                ori_xyz[3 * (size_t)k] = body[i].x; ori_xyz[3 * (size_t)k + 1] = body[i].y; ori_xyz[3 * (size_t)k + 2] = body[i].z;
            }
            if (normvec) memcpy(normvec + 4 * (size_t)k, &nv[i], 16);
        }
        k++;
    }
    *m = k;
    return LIINIT_OK;
}

int liinit_map_incremental(liinit_ctx* h, const double* R, const double* p, const double* RLI, const double* TLI, double ds,
                           int flg_EKF_inited, int* n_add, int* n_nod) {
    if (!h || !R || !p || !RLI || !TLI) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    int n = c->scan_n;
    if (n <= 0) return fail(c, LIINIT_ERR_INVALID, "no scan uploaded");
    materialize_scan(c);
    {
        int r = init_scan_state(c);   // no search pass on this scan yet: every point has "no neighbours" (-> PointToAdd)
        if (r) return r;
        // N > 1: the Nearest_Points of the other ranks' shards; then every rank applies the WHOLE frame's update to its replica
        r = gather_scan_state(c);
        if (r) return r;
    }
    c->map_epoch++;
    c->map_version++;
    {
        int r = maybe_compact(c, n);
        if (r) return r;
    }
    PoseD P;
    fill_pose(P, R, p, RLI, TLI);
    static const int zeros[2] = {0, 0};
    CU(cudaMemcpyAsync(c->d_counters + CNT_NADD, zeros, 2 * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    k_incr_classify<<<nblk(n, 256), 256, 0, c->stream>>>(c->M, P, c->d_body, n, c->d_near_xyz, ds, flg_EKF_inited, c->d_world,
                                                        c->d_flag);
    c->launches++;
    CU(cudaGetLastError());
    // Add_Points(PointToAdd, true) then Add_Points(PointNoNeedDownsample, false) (laserMapping.cpp:556-557).
    // d_world (float4) is the point source; it stays untouched by the inserts.
    int r = downsample_insert(c, c->d_world, n, c->d_flag, 1);
    if (r) return r;
    r = plain_insert(c, c->d_world, n, c->d_flag, 2);
    if (r) return r;
    r = fetch_counters(c);
    if (r) return r;
    if (n_add) *n_add = c->h_counters[CNT_NADD];
    if (n_nod) *n_nod = c->h_counters[CNT_NNOD];
    return check_map_err(c);
}

int liinit_last_pass_timing(liinit_ctx* h, float* kernel_ms, int* launches) {
    if (!h) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    CU(cudaEventSynchronize(c->ev1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    c->last_ms = ms;
    if (kernel_ms) *kernel_ms = ms;
    if (launches) *launches = c->last_launches;
    return LIINIT_OK;
}

int liinit_last_pass_kernel_times(liinit_ctx* h, float* knn_ms, float* plane_ms) {
    if (!h) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    CU(cudaEventSynchronize(c->ev1));
    float a = 0.f, b = 0.f;
    if (c->last_was_search) {
        CU(cudaEventElapsedTime(&a, c->ev0, c->evm));
        CU(cudaEventElapsedTime(&b, c->evm, c->ev1));
    } else {
        CU(cudaEventElapsedTime(&b, c->ev0, c->ev1));
    }
    if (knn_ms) *knn_ms = a;
    if (plane_ms) *plane_ms = b;
    return LIINIT_OK;
}

int liinit_debug_esti_plane(liinit_ctx* h, const float* nb_xyz, int n, double* pabcd, unsigned char* valid) {
    if (!h || !nb_xyz || !pabcd || !valid || n < 0) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    CU(cudaSetDevice(c->device));
    if (n == 0) return LIINIT_OK;
    float* d_in = nullptr;
    double* d_out = nullptr;
    unsigned char* d_ok = nullptr;
    int rc = LIINIT_OK;
    if (cudaMalloc(&d_in, (size_t)n * 15 * 4) != cudaSuccess || cudaMalloc(&d_out, (size_t)n * 32) != cudaSuccess || cudaMalloc(&d_ok, (size_t)n) != cudaSuccess) {
        rc = fail(c, LIINIT_ERR_CUDA, "cudaMalloc (debug_esti_plane)");
    } else {
        cudaMemcpyAsync(d_in, nb_xyz, (size_t)n * 15 * 4, cudaMemcpyHostToDevice, c->stream);
        k_debug_esti_plane<<<nblk(n, 128), 128, 0, c->stream>>>(d_in, n, d_out, d_ok);
        c->launches++;
        cudaMemcpyAsync(pabcd, d_out, (size_t)n * 32, cudaMemcpyDeviceToHost, c->stream);
        cudaMemcpyAsync(valid, d_ok, (size_t)n, cudaMemcpyDeviceToHost, c->stream);
        cudaError_t e = cudaStreamSynchronize(c->stream);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) rc = fail(c, LIINIT_ERR_CUDA, std::string("debug_esti_plane: ") + cudaGetErrorString(e));
    }
    cudaFree(d_in); cudaFree(d_out); cudaFree(d_ok);
    return rc;
}

// ---- multi-GPU (SURVEY.md section 8e) -----------------------------------------------------------------------
int liinit_comm_unique_id(void* id128) {
    if (!id128) return LIINIT_ERR_INVALID;
#ifdef LI_SIMT_EMUL
    return LIINIT_ERR_INVALID;
#else
    NcclApi* N = nccl_api();
    if (!N) {
        g_create_error = "NCCL is not available (dlopen libnccl.so.2 failed)";
        return LIINIT_ERR_CUDA;
    }
    static_assert(sizeof(ncclUniqueId) == LIINIT_COMM_ID_BYTES, "ncclUniqueId size");
    ncclUniqueId id;
    ncclResult_t nr = N->GetUniqueId(&id);
    if (nr != ncclSuccess) {
        g_create_error = std::string("ncclGetUniqueId: ") + N->GetErrorString(nr);
        return LIINIT_ERR_CUDA;
    }
    memcpy(id128, &id, sizeof(id));
    return LIINIT_OK;
#endif
}

int liinit_comm_init(liinit_ctx* h, const void* id128, int nranks, int rank) {
    if (!h || !id128 || nranks < 1 || nranks > 64 || rank < 0 || rank >= nranks) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
#ifdef LI_SIMT_EMUL
    return fail(c, LIINIT_ERR_INVALID, "no communicator in the CPU checker");
#else
    CU(cudaSetDevice(c->device));
    if (c->comm) return fail(c, LIINIT_ERR_INVALID, "communicator already attached");
    NcclApi* N = nccl_api();
    if (!N) return fail(c, LIINIT_ERR_CUDA, "NCCL is not available (dlopen libnccl.so.2 failed)");
    CU(cudaStreamSynchronize(c->stream));
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    ncclResult_t nr = N->CommInitRank(&c->comm, nranks, id, rank);
    if (nr != ncclSuccess) {
        c->comm = nullptr;
        return fail(c, LIINIT_ERR_CUDA, std::string("ncclCommInitRank: ") + N->GetErrorString(nr));
    }
    c->nranks = nranks;
    c->rank = rank;
    if (c->scan_n > 0) set_scan(c, c->scan_n);   // re-cut a frame that is already resident
    // ---- peer-memory exchange (one process per GPU on one NVLink node): every rank's buffer mapped into every process through CUDA IPC.
    // If any rank cannot set it up (same process, no peer access, LIINIT_COMM_MODE=nccl), ALL ranks stay on ncclAllReduce.
    c->comm_p2p = false;
    if (nranks > 1) {
        const char* mode = getenv("LIINIT_COMM_MODE");
        int ok = !(mode && !strcmp(mode, "nccl")) ? 1 : 0;
        const size_t blk_bytes = (size_t)2 * nranks * 160 * sizeof(double), flag_bytes = (size_t)2 * nranks * sizeof(unsigned);
        cudaIpcMemHandle_t mine;
        memset(&mine, 0, sizeof(mine));
        if (ok && (cudaMalloc(&c->d_xbuf, blk_bytes + flag_bytes) != cudaSuccess || cudaMemset(c->d_xbuf, 0, blk_bytes + flag_bytes) != cudaSuccess ||
                   cudaIpcGetMemHandle(&mine, c->d_xbuf) != cudaSuccess)) {
            ok = 0;
            cudaGetLastError();
        }
        // all-gather of the 64-byte handles (+ a 4-byte "fine so far" word) through the communicator that now exists
        const size_t rec = sizeof(cudaIpcMemHandle_t) + 8;
        DevBuf<unsigned char> dh;
        std::vector<unsigned char> hh(rec * nranks, 0);
        if (dh.alloc(rec * nranks) != cudaSuccess) return fail(c, LIINIT_ERR_CUDA, "cudaMalloc (comm handles)");
        memcpy(hh.data() + rec * rank, &mine, sizeof(mine));
        memcpy(hh.data() + rec * rank + sizeof(mine), &ok, sizeof(int));
        CU(cudaMemcpy(dh.p + rec * rank, hh.data() + rec * rank, rec, cudaMemcpyHostToDevice));
        nr = N->AllGather(dh.p + rec * rank, dh.p, rec, ncclChar, c->comm, c->stream);
        if (nr != ncclSuccess) return fail(c, LIINIT_ERR_CUDA, std::string("ncclAllGather (comm handles): ") + N->GetErrorString(nr));
        CU(cudaStreamSynchronize(c->stream));
        CU(cudaMemcpy(hh.data(), dh.p, rec * nranks, cudaMemcpyDeviceToHost));
        for (int r = 0; r < nranks; r++) {
            int okr = 0;
            memcpy(&okr, hh.data() + rec * r + sizeof(mine), sizeof(int));
            ok = ok && okr;
        }
        XchgTable T;
        memset(&T, 0, sizeof(T));
        if (ok) {
            for (int r = 0; r < nranks && ok; r++) {
                void* base = c->d_xbuf;
                if (r != rank) {
                    cudaIpcMemHandle_t hr;
                    memcpy(&hr, hh.data() + rec * r, sizeof(hr));
                    if (cudaIpcOpenMemHandle(&base, hr, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                        ok = 0;
                        cudaGetLastError();
                        break;
                    }
                    c->peer_map[r] = base;
                }
                T.blocks[r] = (double*)base;
                T.flags[r] = (unsigned*)((unsigned char*)base + blk_bytes);
            }
        }
        // second agreement: did every rank open every handle? (sum of the failures over the ranks)
        {
            DevBuf<double> dv;
            if (dv.alloc(1) != cudaSuccess) return fail(c, LIINIT_ERR_CUDA, "cudaMalloc (comm agreement)");
            double bad = ok ? 0.0 : 1.0;
            CU(cudaMemcpy(dv.p, &bad, sizeof(double), cudaMemcpyHostToDevice));
            nr = N->AllReduce(dv.p, dv.p, 1, ncclDouble, ncclSum, c->comm, c->stream);
            if (nr != ncclSuccess) return fail(c, LIINIT_ERR_CUDA, std::string("ncclAllReduce (comm agreement): ") + N->GetErrorString(nr));
            CU(cudaStreamSynchronize(c->stream));
            CU(cudaMemcpy(&bad, dv.p, sizeof(double), cudaMemcpyDeviceToHost));
            ok = bad == 0.0;
        }
        if (ok) {
            T.local = c->d_acc;
            T.nranks = nranks;
            T.rank = rank;
            CU(cudaMalloc(&c->d_xtab, sizeof(XchgTable)));
            CU(cudaMemcpy(c->d_xtab, &T, sizeof(T), cudaMemcpyHostToDevice));
            c->comm_p2p = true;
            c->xseq = 0;
        }
    }
    return LIINIT_OK;
#endif
}

int liinit_comm_last_local(liinit_ctx* h, double* out160) {
    if (!h || !out160) return LIINIT_ERR_INVALID;
    Ctx* c = &h->c;
    if (c->nranks <= 1) return fail(c, LIINIT_ERR_INVALID, "no communicator attached");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaMemcpy(out160, c->d_acc, 160 * sizeof(double), cudaMemcpyDeviceToHost));
    return LIINIT_OK;
}

int liinit_comm_mode(liinit_ctx* h, int* peer_memory) {
    if (!h || !peer_memory) return LIINIT_ERR_INVALID;
    *peer_memory = (h->c.nranks > 1 && h->c.comm_p2p) ? 1 : 0;
    return LIINIT_OK;
}

int liinit_comm_info(liinit_ctx* h, int* nranks, int* rank, int* shard_lo, int* shard_n) {
    if (!h) return LIINIT_ERR_INVALID;
    if (nranks) *nranks = h->c.nranks;
    if (rank) *rank = h->c.rank;
    if (shard_lo) *shard_lo = h->c.shard_lo;
    if (shard_n) *shard_n = h->c.S.n;
    return LIINIT_OK;
}

int liinit_set_reseed(liinit_ctx* h, int enabled) {
    if (!h) return LIINIT_ERR_INVALID;
    h->c.reseed = enabled != 0;
    return LIINIT_OK;
}

int liinit_knn_index(liinit_ctx* h, int* knn_index) {
    if (!h || !knn_index) return LIINIT_ERR_INVALID;
    *knn_index = h->c.cells ? LIINIT_KNN_CELLS : LIINIT_KNN_BRICKS;
    return LIINIT_OK;
}

int liinit_launch_count(liinit_ctx* h, long long* launches) {
    if (!h || !launches) return LIINIT_ERR_INVALID;
    *launches = h->c.launches;
    return LIINIT_OK;
}

}  // extern "C"
