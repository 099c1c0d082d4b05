// Host side of single linkage: label the sorted edges of a minimum spanning tree into scipy's linkage
// matrix Z (engine.single_linkage_host).  Single linkage merges, at every height, the two clusters the
// next MST edge joins, so the dendrogram is a union-find over the edges in order: O(N alpha(N)), fast at
// 10^6 nodes where a Python loop is not.
#include <stdint.h>
#include <cmath>
#include <vector>
#include "../../include/hsd_b200.h"

namespace hsd {
void set_error(const char* fmt, ...);
}

namespace {

int find_root(std::vector<int32_t>& parent, int32_t x) {
    int32_t r = x;
    while (parent[r] != r) r = parent[r];
    while (parent[x] != r) {                                   // path compression
        const int32_t next = parent[x];
        parent[x] = r;
        x = next;
    }
    return r;
}

}  // namespace

extern "C" int hsd_single_linkage_host(const int32_t* u, const int32_t* v, const float* dist, int32_t n, double* Z) {
    if (n < 0) {
        hsd::set_error("%s: %s", __func__, "bad sizes (n must be >= 0)");
        return HSD_ERR_INVALID;
    }
    if (n < 2) return HSD_OK;
    if (!u || !v || !dist || !Z) {
        hsd::set_error("%s: %s", __func__, "null pointer");
        return HSD_ERR_INVALID;
    }
    std::vector<int32_t> parent(n), size(n, 1);
    std::vector<int64_t> cluster(n);                           // cluster id of each union-find root
    for (int32_t i = 0; i < n; ++i) {
        parent[i] = i;
        cluster[i] = i;
    }
    for (int64_t t = 0; t < n - 1; ++t) {
        const int32_t a = u[t], b = v[t];
        const float d = dist[t];
        if (a < 0 || a >= n || b < 0 || b >= n || a == b) {
            hsd::set_error("%s: edge %lld (%d, %d) is not a pair of distinct nodes in 0..n-1", __func__,
                           (long long)t, a, b);
            return HSD_ERR_INVALID;
        }
        if (!std::isfinite(d) || d < 0.f || (t > 0 && d < dist[t - 1])) {
            hsd::set_error("%s: edge %lld: heights must be finite, >= 0 and non-decreasing", __func__, (long long)t);
            return HSD_ERR_INVALID;
        }
        const int32_t ra = find_root(parent, a), rb = find_root(parent, b);
        if (ra == rb) {
            hsd::set_error("%s: edge %lld (%d, %d) closes a cycle: not a spanning tree", __func__, (long long)t, a, b);
            return HSD_ERR_INVALID;
        }
        const int64_t ca = cluster[ra], cb = cluster[rb];
        double* z = Z + 4 * t;
        z[0] = (double)(ca < cb ? ca : cb);
        z[1] = (double)(ca < cb ? cb : ca);
        z[2] = (double)d;
        z[3] = (double)(size[ra] + size[rb]);
        const int32_t big = size[ra] >= size[rb] ? ra : rb, small = big == ra ? rb : ra;   // union by size
        parent[small] = big;
        size[big] += size[small];
        cluster[big] = n + t;
    }
    return HSD_OK;
}
