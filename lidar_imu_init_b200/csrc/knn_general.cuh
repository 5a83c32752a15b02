// knn_general.cuh -- KD_TREE::Nearest_Search(point, k, ..., max_dist) for any 1 <= k <= 32 and any max_dist >= 0 or +INFINITY
// (ikd_Tree.cpp:349-379, Search :825-968) on the brick hash. The k = 5 / max_dist = 5 kernels of the ICP pass (knn_kernels.cuh,
// cells.cuh) are not touched; this header only calls their helpers. DESIGN.md section 3d.
//
// One warp per query. The k best candidates so far are a warp-wide sorted list, one entry per lane (lane i = rank i); a candidate is
// inserted by one ballot (its rank) and one shuffle-up. The k-th distance `kth` is warp-uniform, never grows, and is the candidate
// threshold and the brick prune (INFINITY while fewer than k are known).
//
// Shells on the brick-box distance dbox, as knn5_lockstep, with k for 5 and cap = the largest float not above max_dist for 5:
//     invariant: every brick with dbox < lo2 has been scanned (or could not hold a candidate below kth)
//     step:      scan the bricks with lo2 <= dbox < hi2 (dbox <= cap in the last shell); stop when k are known and kth <= hi2, or when
//                the shell reached cap; otherwise lo2 = hi2 and hi2 = kth (k known: one closing shell) or 4 * hi2, both capped by cap.
// A shell's enumeration box grows with the cube of its radius. When it would hold more bricks than the map has, or leaves the range
// brick keys can pack (LI_CELL_LIMIT: also every query that cannot be packed itself), the rest of the search walks the list of the map's
// bricks instead (`occ`: copies of their hash entries, rebuilt when the map changed): exact, O(bricks) for such a query.
//
// Semantics (include/liinit_gpu.h): point test d2 <= max_dist (ikd_Tree.cpp:842, sic) as d2 <= cap; fp32 (dx*dx+dy*dy)+dz*dz without
// FMA; ascending output in PointType_CMP order (ikd_Tree.h:57-60: |d_a - d_b| < 1e-10 -> smaller x first), applied here on the device.
// The reference's box prune at max_dist^2 (:827-828) is not applied: for max_dist >= 1 it never removes a point that passes the point
// test, below 1 its answer depends on the tree's shape (DESIGN.md section 4, deviations).
#pragma once
#include "knn_kernels.cuh"

#define LI_KNN_GEN_THREADS 256

// Squared distance from the query to brick (kx, ky, kz), a lower bound of every stored point's distance (the rounding slack of
// knn5_lockstep: margin on the box, 1e-6 relative on the result).
__device__ __forceinline__ float li_gen_dbox(const KnnGeom& g, int kx, int ky, int kz, float qx, float qy, float qz) {
    const float lox = (float)li_shl(kx, g.bs) * g.ds - g.margin, hix = (float)li_shl(kx + 1, g.bs) * g.ds + g.margin;
    const float loy = (float)li_shl(ky, g.bs) * g.ds - g.margin, hiy = (float)li_shl(ky + 1, g.bs) * g.ds + g.margin;
    const float loz = (float)li_shl(kz, g.bs) * g.ds - g.margin, hiz = (float)li_shl(kz + 1, g.bs) * g.ds + g.margin;
    const float ex = fmaxf(0.f, fmaxf(lox - qx, qx - hix));
    const float ey = fmaxf(0.f, fmaxf(loy - qy, qy - hiy));
    const float ez = fmaxf(0.f, fmaxf(loz - qz, qz - hiz));
    return (ex * ex + ey * ey + ez * ez) * (1.0f - 1e-6f);
}

// The warp's sorted top-k: lane i holds rank i (d, pool offset) for i < cnt; cnt and kth are warp-uniform.
struct GenTop {
    float d;
    int id;
    int cnt;
    float kth;
};

// Insert (d, id), d < top.kth. Ties keep arrival order (the new entry goes after the equal ones).
__device__ __forceinline__ void li_gen_insert(GenTop& t, int k, float d, int id, int lane) {
    const int pos = __popc(__ballot_sync(LI_FULL, lane < t.cnt && t.d <= d));
    const float ud = __shfl_up_sync(LI_FULL, t.d, 1);
    const int ui = __shfl_up_sync(LI_FULL, t.id, 1);
    if (lane == pos) {
        t.d = d;
        t.id = id;
    } else if (lane > pos) {
        t.d = ud;
        t.id = ui;
    }
    t.cnt = min(t.cnt + 1, k);
    const float last = __shfl_sync(LI_FULL, t.d, k - 1);
    t.kth = (t.cnt == k) ? last : INFINITY;
}

// Scan one slab [f, f + c) (warp-uniform): 32 points per step, the candidates of a step are inserted one after the other.
__device__ __forceinline__ void li_gen_scan(const float4* __restrict__ pool, unsigned f, unsigned c, float qx, float qy, float qz, float cap,
                                            GenTop& t, int k, int lane) {
    for (unsigned j = 0; j < c; j += 32) {
        const bool in = j + (unsigned)lane < c;
        float d = INFINITY;
        if (in) {
            const float4 p = __ldg(&pool[f + j + lane]);
            d = li_dist2(qx, qy, qz, p.x, p.y, p.z);
        }
        unsigned m = __ballot_sync(LI_FULL, in && d <= cap && d < t.kth);
        while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            const float dd = __shfl_sync(LI_FULL, d, src);
            if (dd < t.kth) li_gen_insert(t, k, dd, (int)(f + j + src), lane);
        }
    }
}

// Scan the bricks found by this step's probes (bit l of fm: lane l found one, its slab in (first, count)).
__device__ __forceinline__ void li_gen_scan_found(const float4* __restrict__ pool, unsigned fm, unsigned first, unsigned count, float qx, float qy,
                                                  float qz, float cap, GenTop& t, int k, int lane) {
    while (fm) {
        const int src = __ffs(fm) - 1;
        fm &= fm - 1;
        const unsigned f = __shfl_sync(LI_FULL, first, src), c = __shfl_sync(LI_FULL, count, src);
        li_gen_scan(pool, f, c, qx, qy, qz, cap, t, k, lane);
    }
}

// Exact k-NN of one finite query by the whole warp. occ[0..nb): the map's bricks as copies of their hash entries.
__device__ __forceinline__ void li_gen_search(const MapDev& M, const uint4* __restrict__ occ, int nb, float rho2, float cap, float qx, float qy, float qz,
                                              GenTop& t, int k, int lane) {
    KnnGeom g;
    g.bs = M.bshift;
    g.ds = M.ds;
    const int bc = 1 << g.bs;
    const float inv_ds = 1.0f / g.ds;
    const float aq = fabsf(qx) + fabsf(qy) + fabsf(qz);
    g.margin = 1e-6f * (aq + 16.0f * (float)bc * g.ds);
    const float slk = 0.02f + 4e-7f * aq * inv_ds;
    const float lim = (float)(LI_CELL_LIMIT - 16 * bc);   // cell coordinates whose bricks can be packed, with room for the slack
    float lo2 = 0.f, hi2 = fminf(rho2, cap);
    bool walk = false;   // the rest of the search walks occ
    for (;;) {
        const bool last = hi2 >= cap;
        const float r = sqrtf(hi2) * (1.0f + 1e-6f) + g.margin;
        const float fx0 = floorf((qx - r) * inv_ds - slk), fx1 = floorf((qx + r) * inv_ds + slk);
        const float fy0 = floorf((qy - r) * inv_ds - slk), fy1 = floorf((qy + r) * inv_ds + slk);
        const float fz0 = floorf((qz - r) * inv_ds - slk), fz1 = floorf((qz + r) * inv_ds + slk);
        if (!(fx0 > -lim && fx1 < lim && fy0 > -lim && fy1 < lim && fz0 > -lim && fz1 < lim)) {   // (also NaN-safe)
            walk = true;
            break;
        }
        const int lx = (int)fx0 >> g.bs, hx = (int)fx1 >> g.bs;
        const int ly = (int)fy0 >> g.bs, hy = (int)fy1 >> g.bs;
        const int lz = (int)fz0 >> g.bs, hz = (int)fz1 >> g.bs;
        const int nx = hx - lx + 1, ny = hy - ly + 1, nz = hz - lz + 1;
        if ((float)nx * (float)ny * (float)nz > (float)nb) {
            walk = true;
            break;
        }
        const int nxy = nx * ny, total = nxy * nz;
        for (int base = 0; base < total; base += 32) {
            const int idx = base + lane;
            bool found = false;
            unsigned first = 0, count = 0;
            if (idx < total) {
                const int iz = idx / nxy, rem = idx - iz * nxy;
                const int iy = rem / nx, ix = rem - iy * nx;
                const int kx = lx + ix, ky = ly + iy, kz = lz + iz;
                const float dbox = li_gen_dbox(g, kx, ky, kz, qx, qy, qz);
                if (dbox >= lo2 && (last ? dbox <= cap : dbox < hi2) && dbox < t.kth) {
                    const unsigned long long key = li_pack_key(kx, ky, kz);
                    unsigned h;
                    const uint4 e = li_brick_probe_issue(M.ent, M.mask, key, h);
                    found = li_brick_probe_finish(M.ent, M.mask, key, h, e, first, count) && count > 0u;
                }
            }
            li_gen_scan_found(M.pool, __ballot_sync(LI_FULL, found), first, count, qx, qy, qz, cap, t, k, lane);
        }
        const bool full = t.cnt == k;
        if (last || (full && t.kth <= hi2)) break;
        lo2 = hi2;
        hi2 = full ? fminf(t.kth * (1.0f + 1e-6f), cap) : fminf(4.0f * hi2, cap);
    }
    if (!walk) return;
    for (int base = 0; base < nb; base += 32) {
        const int i = base + lane;
        bool found = false;
        unsigned first = 0, count = 0;
        if (i < nb) {
            const uint4 e = __ldg(&occ[i]);
            const unsigned long long key = (unsigned long long)e.x | ((unsigned long long)e.y << 32);
            const int kx = (int)(unsigned)(key >> 42) - LI_CELL_LIMIT, ky = (int)((unsigned)(key >> 21) & 0x1fffffu) - LI_CELL_LIMIT,
                      kz = (int)((unsigned)key & 0x1fffffu) - LI_CELL_LIMIT;
            const float dbox = li_gen_dbox(g, kx, ky, kz, qx, qy, qz);
            found = e.w > 0u && dbox >= lo2 && dbox <= cap && dbox < t.kth;
            first = e.z;
            count = e.w;
        }
        li_gen_scan_found(M.pool, __ballot_sync(LI_FULL, found), first, count, qx, qy, qz, cap, t, k, lane);
    }
}

// occ[i] = hash entry of brick i (M.brick_slots order) for i < counters[CNT_BRICKS]; the count is read on the device.
__global__ void k_knn_occ_build(MapDev M, uint4* __restrict__ occ) {
    const int nb = M.counters[CNT_BRICKS];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nb; i += gridDim.x * blockDim.x) occ[i] = M.ent[M.brick_slots[i]];
}

// n queries at q[i * stride + 0..2]; out_xyz [n*k*3], out_d2 [n*k] (-1 / zero xyz past the count), out_cnt [n].
__global__ void __launch_bounds__(LI_KNN_GEN_THREADS) k_knn_general(MapDev M, const uint4* __restrict__ occ, const float* __restrict__ q, int stride,
                                                                    int n, int k, float cap, float rho2, float* __restrict__ out_xyz,
                                                                    float* __restrict__ out_d2, int* __restrict__ out_cnt) {
    const int lane = threadIdx.x & 31;
    const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    const int nb = M.counters[CNT_BRICKS];
    for (int qi = warp_global; qi < n; qi += nwarps) {   // warp-uniform
        const float* qp = q + (size_t)qi * stride;
        const float qx = qp[0], qy = qp[1], qz = qp[2];
        GenTop t;
        t.d = INFINITY;
        t.id = -1;
        t.cnt = 0;
        t.kth = INFINITY;
        if (isfinite(qx) && isfinite(qy) && isfinite(qz)) li_gen_search(M, occ, nb, rho2, cap, qx, qy, qz, t, k, lane);
        float px = 0.f, py = 0.f, pz = 0.f;
        if (lane < t.cnt) {
            const float4 p = __ldg(&M.pool[t.id]);
            px = p.x;
            py = p.y;
            pz = p.z;
        }
        // PointType_CMP order: entries whose distances differ by less than 1e-10 go by ascending x (odd-even transposition, k rounds)
        for (int pass = 0; pass < t.cnt; pass++) {
            const bool lower = ((lane ^ pass) & 1) == 0;
            const int partner = lower ? lane + 1 : lane - 1;
            const float od = __shfl_sync(LI_FULL, t.d, partner & 31);
            const float ox = __shfl_sync(LI_FULL, px, partner & 31);
            const float oy = __shfl_sync(LI_FULL, py, partner & 31);
            const float oz = __shfl_sync(LI_FULL, pz, partner & 31);
            const bool pair = lane < t.cnt && partner >= 0 && partner < t.cnt;
            if (pair && fabsf(t.d - od) < 1e-10f && (lower ? ox < px : px < ox)) {
                t.d = od;
                px = ox;
                py = oy;
                pz = oz;
            }
        }
        if (lane < k) {
            const size_t o = (size_t)qi * k + lane;
            const bool have = lane < t.cnt;
            out_d2[o] = have ? t.d : -1.f;
            out_xyz[3 * o] = px;
            out_xyz[3 * o + 1] = py;
            out_xyz[3 * o + 2] = pz;
        }
        if (lane == 0) out_cnt[qi] = t.cnt;
    }
}
