// liinit_adapter.hpp -- header-only C++ adapter with the method names of the reference's KD_TREE
// (include/ikd-Tree/ikd_Tree.h:165-187) over the C-ABI, templated on the point type so that it binds to
// pcl::PointXYZINormal (48 bytes, x/y/z first) without this repository depending on PCL. INTEGRATION.md shows
// the node-side patch. Errors become exceptions here (the C-ABI itself never throws).
#pragma once
#include <stdexcept>
#include <string>
#include <vector>

#include "liinit_gpu.h"

namespace liinit {

template <class PointT, class Alloc = std::allocator<PointT>>
class DeviceMap {
public:
    using PointVector = std::vector<PointT, Alloc>;
    static_assert(sizeof(PointT) % sizeof(float) == 0, "point type must be made of floats");

    explicit DeviceMap(const liinit_config& cfg) {
        if (liinit_create(&cfg, &h_) != LIINIT_OK) throw std::runtime_error(std::string("liinit_create: ") + liinit_last_error(nullptr));
    }
    ~DeviceMap() { liinit_destroy(h_); }
    DeviceMap(const DeviceMap&) = delete;
    DeviceMap& operator=(const DeviceMap&) = delete;

    liinit_ctx* ctx() { return h_; }

    // KD_TREE::Build(PointVector) (ikd_Tree.cpp:336-347)
    void Build(const PointVector& pts) { ck(liinit_map_build(h_, fptr(pts), stride(), (int)pts.size())); }
    // KD_TREE::Add_Points(PointVector&, bool) (ikd_Tree.cpp:381-456)
    int Add_Points(const PointVector& pts, bool downsample_on) {
        int added = 0;
        if (!pts.empty()) ck(liinit_map_add_points(h_, fptr(pts), stride(), (int)pts.size(), downsample_on ? 1 : 0, &added));
        return added;
    }
    // KD_TREE::size / validnum (ikd_Tree.cpp:71-88,120-137)
    int size() { int n = 0; ck(liinit_map_size(h_, &n)); return n; }
    int validnum() { int n = 0; ck(liinit_map_validnum(h_, &n)); return n; }
    // KD_TREE::Nearest_Search(point, k, Nearest_Points, Point_Distance, max_dist) (ikd_Tree.cpp:349-379) for one query, 1 <= k <= 32.
    // k = 5 with max_dist = 5 (the node's call, laserMapping.cpp:980) takes the path of the ICP pass; any other k / max_dist the general
    // search (liinit_map_knn_search). The reference's default max_dist is INFINITY (ikd_Tree.h:176); this one stays 5 for existing callers.
    void Nearest_Search(const PointT& p, int k, PointVector& near, std::vector<float>& d2, double max_dist = 5.0) {
        float q[3] = {p.x, p.y, p.z}, xyz[3 * LIINIT_KNN_MAX_K], dd[LIINIT_KNN_MAX_K];
        int cnt = 0;
        if (k == LIINIT_NUM_MATCH_POINTS && max_dist == 5.0) ck(liinit_map_nearest_search(h_, q, 3, 1, max_dist, xyz, dd, &cnt));
        else ck(liinit_map_knn_search(h_, q, 3, 1, k, max_dist, xyz, dd, &cnt));
        near.assign(cnt, PointT());
        d2.assign(dd, dd + cnt);
        for (int j = 0; j < cnt; j++) { near[j].x = xyz[3 * j]; near[j].y = xyz[3 * j + 1]; near[j].z = xyz[3 * j + 2]; }
    }
    // feats_down_body upload (laserMapping.cpp:917-919)
    void UploadScan(const PointVector& body) { ck(liinit_scan_upload(h_, fptr(body), stride(), (int)body.size())); }
    // body must live in page-locked memory (cudaHostRegister on the vector's storage) and stay untouched until the
    // first search pass of the scan has returned: the search kernel reads it in place, no staging copy.
    void AttachScan(const PointVector& body) { ck(liinit_scan_attach_host(h_, fptr(body), stride(), (int)body.size())); }

private:
    static int stride() { return (int)(sizeof(PointT) / sizeof(float)); }
    static const float* fptr(const PointVector& v) { return reinterpret_cast<const float*>(v.data()); }
    void ck(int rc) {
        if (rc != LIINIT_OK) throw std::runtime_error(std::string("liinit: ") + liinit_last_error(h_));
    }
    liinit_ctx* h_ = nullptr;
};

}  // namespace liinit
