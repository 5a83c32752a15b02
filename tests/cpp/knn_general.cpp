// tests/cpp/knn_general.cpp -- TEST: KD_TREE::Nearest_Search with the reference's default max_dist (INFINITY, ikd_Tree.h:176) and
// k = 10 through the C++ adapter (liinit_adapter.hpp) with the reference's point type, one query per call, as a node would call it.
// tests/test_knn_general.py compiles it on the CPU (-std=c++14 -Wall -Werror) and, on a GPU, compares what it writes with the
// ctypes path (liinit_map_knn_search) on the same inputs.
//   usage: knn_general <in.bin> <out.bin>
//   in : int32 n_map, n_query; float32 ds; float32 map[n_map*3], query[n_query*3]
//   out: per query int32 count; float32 xyz[10*3], d2[10] (zeros / -1 past the count)
#include <pcl/point_types.h>
#include <Eigen/StdVector>

#include <cmath>
#include <cstdio>
#include <vector>

#include "liinit_adapter.hpp"

typedef pcl::PointXYZINormal PointType;                                            // include/common_lib.h:37
typedef std::vector<PointType, Eigen::aligned_allocator<PointType>> PointVector;   // include/common_lib.h:41

static bool rd(FILE* f, void* p, size_t n) { return fread(p, 1, n, f) == n; }

int main(int argc, char** argv) {
    if (argc < 3) return 2;
    FILE* f = fopen(argv[1], "rb");
    if (!f) return 2;
    int hdr[2];
    float ds = 0.f;
    if (!rd(f, hdr, sizeof(hdr)) || !rd(f, &ds, sizeof(ds))) return 2;
    std::vector<float> mp((size_t)hdr[0] * 3), qs((size_t)hdr[1] * 3);
    if (!rd(f, mp.data(), mp.size() * 4) || !rd(f, qs.data(), qs.size() * 4)) return 2;
    fclose(f);
    PointVector map_pts(hdr[0]);
    for (int i = 0; i < hdr[0]; i++) {
        map_pts[i].x = mp[3 * i];
        map_pts[i].y = mp[3 * i + 1];
        map_pts[i].z = mp[3 * i + 2];
    }
    liinit_config cfg = {};
    cfg.filter_size_map = ds;
    cfg.max_map_points = hdr[0] * 2 + 100000;
    cfg.max_scan_points = 1000;
    liinit::DeviceMap<PointType, Eigen::aligned_allocator<PointType>> tree(cfg);
    tree.Build(map_pts);
    FILE* o = fopen(argv[2], "wb");
    if (!o) return 2;
    const int K = 10;
    for (int i = 0; i < hdr[1]; i++) {
        PointType p;
        p.x = qs[3 * i];
        p.y = qs[3 * i + 1];
        p.z = qs[3 * i + 2];
        PointVector near;
        std::vector<float> d2;
        tree.Nearest_Search(p, K, near, d2, INFINITY);
        const int cnt = (int)near.size();
        float xyz[3 * K] = {0.f}, dd[K];
        for (int j = 0; j < K; j++) dd[j] = -1.f;
        for (int j = 0; j < cnt; j++) {
            xyz[3 * j] = near[j].x;
            xyz[3 * j + 1] = near[j].y;
            xyz[3 * j + 2] = near[j].z;
            dd[j] = d2[j];
        }
        fwrite(&cnt, 4, 1, o);
        fwrite(xyz, 4, 3 * K, o);
        fwrite(dd, 4, K, o);
    }
    fclose(o);
    return 0;
}
