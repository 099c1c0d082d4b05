// Host side of HDBSCAN: label the single-linkage tree Z of the mutual-reachability MST (hsd_single_linkage_host's
// linkage; engine.hdbscan_host).  A port of scikit-learn 1.9's tree_to_labels (sklearn/cluster/_hdbscan/_tree.pyx,
// BSD-3-Clause) with cluster_selection_epsilon = 0 and max_cluster_size = None: _condense_tree, _compute_stability,
// _get_clusters (eom / leaf, allow_single_cluster), _do_labelling, max_lambdas and get_probabilities.  The condensed
// tree's rows come out in the same order and every float64 operation is the same, in the same order (lambda = 1 / d,
// +inf for d = 0, and the inf - inf = NaN stabilities that follow), so EOM's comparisons are decided identically and
// the labels and probabilities are sklearn's bit for bit.  Flat arrays, O(N alpha(N)): fast at 10^6 nodes, where
// the Python loops of the original are not.
#include <stdint.h>
#include <algorithm>
#include <cmath>
#include <limits>
#include <vector>
#include "../../include/hsd_b200.h"

namespace hsd {
void set_error(const char* fmt, ...);
}

namespace {

struct Condensed {                                              // CONDENSED_dtype, one vector per field
    std::vector<int64_t> parent, child, size;
    std::vector<double> value;
    void push(int64_t p, int64_t c, double v, int64_t s) {
        parent.push_back(p);
        child.push_back(c);
        value.push_back(v);
        size.push_back(s);
    }
};

// _condense_tree: the hierarchy's nodes in breadth-first order from the root (bfs_from_hierarchy's level order is a
// FIFO queue's order); a child smaller than min_cluster_size falls out as its points, in its own breadth-first order.
void condense_tree(const int64_t* left, const int64_t* right, const int64_t* csize, const double* dist, int64_t n,
                   int64_t min_cluster_size, Condensed& t) {
    const int64_t root = 2 * (n - 1);
    std::vector<int64_t> order, sub;
    order.reserve(root + 1);
    order.push_back(root);
    for (size_t h = 0; h < order.size(); ++h) {
        const int64_t x = order[h];
        if (x >= n) {
            order.push_back(left[x - n]);
            order.push_back(right[x - n]);
        }
    }
    std::vector<int64_t> relabel(root + 1, 0);
    std::vector<uint8_t> ignore(root + 1, 0);
    relabel[root] = n;
    int64_t next_label = n + 1;
    auto fall_out = [&](int64_t top, int64_t label, double lambda) {   // every point under top leaves label
        sub.clear();
        sub.push_back(top);
        for (size_t h = 0; h < sub.size(); ++h) {
            const int64_t x = sub[h];
            if (x < n) {
                t.push(label, x, lambda, 1);
            } else {
                sub.push_back(left[x - n]);
                sub.push_back(right[x - n]);
            }
            ignore[x] = 1;
        }
    };
    for (const int64_t node : order) {
        if (ignore[node] || node < n) continue;
        const int64_t l = left[node - n], r = right[node - n];
        const double distance = dist[node - n];
        const double lambda = distance > 0.0 ? 1.0 / distance : std::numeric_limits<double>::infinity();
        const int64_t lc = l >= n ? csize[l - n] : 1, rc = r >= n ? csize[r - n] : 1;
        if (lc >= min_cluster_size && rc >= min_cluster_size) {
            relabel[l] = next_label++;
            t.push(relabel[node], relabel[l], lambda, lc);
            relabel[r] = next_label++;
            t.push(relabel[node], relabel[r], lambda, rc);
        } else if (lc < min_cluster_size && rc < min_cluster_size) {
            fall_out(l, relabel[node], lambda);
            fall_out(r, relabel[node], lambda);
        } else if (lc < min_cluster_size) {
            relabel[r] = relabel[node];
            fall_out(l, relabel[node], lambda);
        } else {
            relabel[l] = relabel[node];
            fall_out(r, relabel[node], lambda);
        }
    }
}

// TreeUnionFind: union by rank, the first argument's root winning ties; find compresses the path
struct UnionFind {
    std::vector<int64_t> parent, rank;
    explicit UnionFind(int64_t size) : parent(size), rank(size, 0) {
        for (int64_t i = 0; i < size; ++i) parent[i] = i;
    }
    int64_t find(int64_t x) {
        int64_t r = x;
        while (parent[r] != r) r = parent[r];
        while (parent[x] != r) {
            const int64_t next = parent[x];
            parent[x] = r;
            x = next;
        }
        return r;
    }
    void unite(int64_t x, int64_t y) {
        const int64_t xr = find(x), yr = find(y);
        if (rank[xr] < rank[yr]) {
            parent[xr] = yr;
        } else if (rank[xr] > rank[yr]) {
            parent[yr] = xr;
        } else {
            parent[yr] = xr;
            rank[xr] += 1;
        }
    }
};

}  // namespace

extern "C" int hsd_hdbscan_host(const double* Z, int32_t n32, int32_t min_cluster_size, int32_t method,
                                int32_t allow_single_cluster, int64_t* labels, double* probabilities) {
    if (n32 < 2) {
        hsd::set_error("%s: %s", __func__, "bad sizes (n must be >= 2)");
        return HSD_ERR_INVALID;
    }
    if (min_cluster_size < 2) {
        hsd::set_error("%s: %s", __func__, "min_cluster_size must be >= 2");
        return HSD_ERR_INVALID;
    }
    if (method != 0 && method != 1) {
        hsd::set_error("%s: %s", __func__, "method must be 0 (eom) or 1 (leaf)");
        return HSD_ERR_INVALID;
    }
    if (!Z || !labels || !probabilities) {
        hsd::set_error("%s: %s", __func__, "null pointer");
        return HSD_ERR_INVALID;
    }
    const int64_t n = n32;
    // Z as HIERARCHY_dtype; a row may only merge nodes formed before it, each once, so the tree is a tree
    std::vector<int64_t> left(n - 1), right(n - 1), csize(n - 1);
    std::vector<double> dist(n - 1);
    std::vector<uint8_t> used(2 * n - 1, 0);
    for (int64_t t = 0; t < n - 1; ++t) {
        const double* z = Z + 4 * t;
        const double lo = z[0], hi = z[1];
        if (!(lo >= 0 && hi >= 0 && lo < (double)(n + t) && hi < (double)(n + t)) || lo == hi ||
            lo != std::floor(lo) || hi != std::floor(hi) || used[(int64_t)lo] || used[(int64_t)hi]) {
            hsd::set_error("%s: row %lld of Z does not merge two distinct unmerged clusters formed before it",
                           __func__, (long long)t);
            return HSD_ERR_INVALID;
        }
        left[t] = (int64_t)lo;
        right[t] = (int64_t)hi;
        used[left[t]] = used[right[t]] = 1;
        const int64_t s = (left[t] >= n ? csize[left[t] - n] : 1) + (right[t] >= n ? csize[right[t] - n] : 1);
        if (z[3] != (double)s) {
            hsd::set_error("%s: row %lld of Z: cluster size %g, its children hold %lld", __func__, (long long)t, z[3],
                           (long long)s);
            return HSD_ERR_INVALID;
        }
        csize[t] = s;
        dist[t] = z[2];
    }

    Condensed t;
    condense_tree(left.data(), right.data(), csize.data(), dist.data(), n, min_cluster_size, t);
    const int64_t rows = (int64_t)t.parent.size();
    const int64_t root = n;                                      // min(parent): the root's label
    int64_t max_parent = root, max_child = root;
    for (int64_t i = 0; i < rows; ++i) {
        max_parent = std::max(max_parent, t.parent[i]);
        max_child = std::max(max_child, t.child[i]);
    }

    // _compute_stability: sum over rows of (lambda - birth(parent)) * size, in row order
    std::vector<double> births(max_child + 1, std::numeric_limits<double>::quiet_NaN());
    for (int64_t i = 0; i < rows; ++i) births[t.child[i]] = t.value[i];
    births[root] = 0.0;
    const int64_t n_clusters = max_parent - root + 1;
    std::vector<double> stability(n_clusters, 0.0);
    for (int64_t i = 0; i < rows; ++i) {
        const int64_t p = t.parent[i];
        stability[p - root] += (t.value[i] - births[p]) * (double)t.size[i];
    }

    // _get_clusters.  The cluster tree is the rows with size > 1; a cluster's children are in row order
    std::vector<int64_t> tree_parent(n_clusters, -1), n_children(n_clusters, 0), child0(n_clusters, -1),
        child1(n_clusters, -1);
    bool any_tree_row = false;
    for (int64_t i = 0; i < rows; ++i) {
        if (t.size[i] <= 1) continue;
        any_tree_row = true;
        const int64_t p = t.parent[i] - root, c = t.child[i] - root;
        tree_parent[c] = p;
        (n_children[p]++ == 0 ? child0 : child1)[p] = c;          // a split makes exactly two
    }
    // node_list: the clusters in descending id (a child's id exceeds its parent's), the root only when a single
    // cluster is allowed
    auto listed = [&](int64_t c) { return c != 0 || allow_single_cluster; };
    std::vector<uint8_t> is_cluster(n_clusters, 0);
    if (method == 0) {                                           // eom
        std::vector<uint8_t> keep(n_clusters, 0);
        for (int64_t c = n_clusters - 1; c >= 0; --c) {
            if (!listed(c)) continue;
            double subtree = 0.0;                                // np.sum over the children, in row order
            if (n_children[c] >= 1) subtree = stability[child0[c]];
            if (n_children[c] == 2) subtree = subtree + stability[child1[c]];
            if (subtree > stability[c]) {
                stability[c] = subtree;
            } else {
                keep[c] = 1;                                     // and every cluster below it is not one
            }
        }
        // a kept cluster stays one unless a listed cluster above it was kept (it was processed later)
        std::vector<uint8_t> below_kept(n_clusters, 0);
        for (int64_t c = 0; c < n_clusters; ++c) {              // parents first
            const int64_t p = tree_parent[c];
            if (p >= 0 && listed(p)) below_kept[c] = keep[p] || below_kept[p];
            is_cluster[c] = listed(c) && keep[c] && !below_kept[c];
        }
    } else {                                                     // leaf: the cluster tree's leaves, none without it
        for (int64_t c = 0; c < n_clusters; ++c) is_cluster[c] = any_tree_row && listed(c) && n_children[c] == 0;
    }
    std::vector<int64_t> cluster_label(n_clusters, -1);         // cluster_map: ascending ids -> 0, 1, ...
    std::vector<int64_t> label_cluster;
    for (int64_t c = 0; c < n_clusters; ++c) {
        if (!is_cluster[c]) continue;
        cluster_label[c] = (int64_t)label_cluster.size();
        label_cluster.push_back(c + root);
    }

    // _do_labelling
    UnionFind uf(max_parent + 1);
    std::vector<double> point_lambda(n, 0.0);
    double root_max_lambda = -std::numeric_limits<double>::infinity();
    for (int64_t i = 0; i < rows; ++i) {
        const int64_t c = t.child[i], p = t.parent[i];
        if (c < n) point_lambda[c] = t.value[i];
        if (p == root) root_max_lambda = std::max(root_max_lambda, t.value[i]);
        if (!(c >= root && is_cluster[c - root])) uf.unite(p, c);
    }
    for (int64_t i = 0; i < n; ++i) {
        const int64_t cluster = uf.find(i);
        int64_t label = -1;
        if (cluster != root) {                                   // a selected cluster: the first row of its
            label = cluster_label[cluster - root];               // component unites into it, and so do the rest
        } else if (label_cluster.size() == 1 && allow_single_cluster) {
            if (point_lambda[i] >= root_max_lambda) label = cluster_label[0];
        }
        labels[i] = label;
    }

    // get_probabilities, with max_lambdas: the maximum lambda of a parent's LAST run of consecutive rows
    std::vector<double> deaths(max_parent + 1, 0.0);
    int64_t current = t.parent[0];
    double max_lambda = t.value[0];
    for (int64_t i = 1; i < rows; ++i) {
        if (t.parent[i] == current) {
            max_lambda = std::max(max_lambda, t.value[i]);
        } else {
            deaths[current] = max_lambda;
            current = t.parent[i];
            max_lambda = t.value[i];
        }
    }
    deaths[current] = max_lambda;
    for (int64_t i = 0; i < n; ++i) probabilities[i] = 0.0;
    for (int64_t i = 0; i < rows; ++i) {
        const int64_t point = t.child[i];
        if (point >= root || labels[point] == -1) continue;
        const double death = deaths[label_cluster[labels[point]]];
        if (death == 0.0 || std::isinf(t.value[i])) {
            probabilities[point] = 1.0;
        } else {
            probabilities[point] = std::min(t.value[i], death) / death;
        }
    }
    return HSD_OK;
}
