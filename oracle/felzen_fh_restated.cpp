// felzen_fh_restated.cpp -- TEST INFRASTRUCTURE ONLY.
//
// The same two C entry points as felzen_ref_shim.cpp (felzen_ref_graph, felzen_ref_image), computed by a
// restatement of the published Felzenszwalb-Huttenlocher segmentation (P. Felzenszwalb, D. Huttenlocher,
// "Efficient Graph-Based Image Segmentation", IJCV 59(2), 2004, and the authors' public C++ code that the
// reference vendors under prim/src/FelzenSegment).  oracle/build_ref.py builds it when no checkout of the
// reference is at hand, so that tests/test_felzenszwalb_ref.py runs from the repository alone.
//
// The arithmetic follows the published code step for step, in the same order and float width:
//   * Gaussian: taps exp(-0.5 (i/sigma)^2), i < ceil(4 sigma) + 1, normalised by 2 sum_{i>0} |m_i| + |m_0|;
//     separable even convolution with clamped borders, each pass writing its output transposed;
//   * edges: for every pixel in row-major order, to (x+1, y), (x, y+1), (x+1, y+1), (x+1, y-1), weight
//     sqrt((dr)^2 + (dg)^2 + (db)^2) of the smoothed float planes;
//   * merge: std::sort by weight, then a != b && w <= thr[a] && w <= thr[b] joins and sets
//     thr[root] = w + c / |root| (thr starts at c / 1); union by rank, path compression;
//   * min-size pass over the sorted edges; components numbered in row-major order of first appearance.
// For distinct edge weights the resulting partition is fixed by the algorithm alone.
#include <algorithm>
#include <cmath>
#include <vector>

namespace {

struct Edge {
    float w;
    int a, b;
};
inline bool operator<(const Edge& x, const Edge& y) { return x.w < y.w; }

class Forest {
public:
    explicit Forest(int n) : parent_(n), rank_(n, 0), size_(n, 1), sets_(n) {
        for (int i = 0; i < n; ++i) parent_[i] = i;
    }
    int find(int x) {
        int y = x;
        while (y != parent_[y]) y = parent_[y];
        parent_[x] = y;
        return y;
    }
    void join(int x, int y) {
        if (rank_[x] > rank_[y]) {
            parent_[y] = x;
            size_[x] += size_[y];
        } else {
            parent_[x] = y;
            size_[y] += size_[x];
            if (rank_[x] == rank_[y]) rank_[y]++;
        }
        sets_--;
    }
    int size(int x) const { return size_[x]; }
    int sets() const { return sets_; }

private:
    std::vector<int> parent_, rank_, size_;
    int sets_;
};

// sorts `edges` in place (the min-size pass then walks them in that order)
void merge_graph(Forest& u, std::vector<Edge>& edges, float c) {
    std::sort(edges.begin(), edges.end());
    std::vector<float> thr((size_t)u.sets(), c / 1);
    for (const Edge& e : edges) {
        int a = u.find(e.a), b = u.find(e.b);
        if (a != b && e.w <= thr[a] && e.w <= thr[b]) {
            u.join(a, b);
            a = u.find(a);
            thr[a] = e.w + c / u.size(a);
        }
    }
}

void merge_small(Forest& u, const std::vector<Edge>& edges, int min_size) {
    for (const Edge& e : edges) {
        int a = u.find(e.a), b = u.find(e.b);
        if (a != b && (u.size(a) < min_size || u.size(b) < min_size)) u.join(a, b);
    }
}

int number_components(Forest& u, int n, int* labels_out) {
    std::vector<int> index((size_t)n, -1);
    int next = 0;
    for (int v = 0; v < n; ++v) {
        int comp = u.find(v);
        if (index[comp] < 0) index[comp] = next++;
        labels_out[v] = index[comp];
    }
    return u.sets() == next ? next : -1;
}

// src is w x h (row-major, x fastest); dst receives the filtered image transposed (h x w becomes w-major rows)
void convolve_even_transposed(const std::vector<float>& src, int w, int h, const std::vector<float>& mask,
                              std::vector<float>& dst) {
    const int len = (int)mask.size();
    dst.assign((size_t)w * h, 0.f);
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            float sum = mask[0] * src[(size_t)y * w + x];
            for (int i = 1; i < len; ++i)
                sum += mask[i] * (src[(size_t)y * w + std::max(x - i, 0)] + src[(size_t)y * w + std::min(x + i, w - 1)]);
            dst[(size_t)x * h + y] = sum;
        }
}

std::vector<float> smooth(const std::vector<float>& src, int w, int h, float sigma) {
    sigma = std::max(sigma, 0.01F);
    const int len = (int)std::ceil(sigma * 4.0) + 1;
    std::vector<float> mask((size_t)len);
    for (int i = 0; i < len; ++i) {
        const float t = i / sigma;
        mask[i] = std::exp(-0.5 * (t * t));
    }
    float sum = 0;
    for (int i = 1; i < len; ++i) sum += std::fabs(mask[i]);
    sum = 2 * sum + std::fabs(mask[0]);
    for (int i = 0; i < len; ++i) mask[i] /= sum;
    std::vector<float> tmp, dst;
    convolve_even_transposed(src, w, h, mask, tmp);   // h x w -> w x h
    convolve_even_transposed(tmp, h, w, mask, dst);   // back to h x w
    return dst;
}

}  // namespace

extern "C" {

int felzen_ref_graph(int n_vertices, int n_edges, const int* a, const int* b, const float* w, float c, int min_size,
                     int* labels_out) {
    std::vector<Edge> edges((size_t)n_edges);
    for (int i = 0; i < n_edges; ++i) edges[i] = Edge{w[i], a[i], b[i]};
    Forest u(n_vertices);
    merge_graph(u, edges, c);
    merge_small(u, edges, min_size);
    return number_components(u, n_vertices, labels_out);
}

int felzen_ref_image(const unsigned char* rgb_in, int h, int w, float sigma, float c, int min_size, int* labels_out) {
    const size_t n = (size_t)w * h;
    std::vector<float> plane[3];
    for (int k = 0; k < 3; ++k) {
        plane[k].resize(n);
        for (size_t i = 0; i < n; ++i) plane[k][i] = rgb_in[i * 3 + k];
        plane[k] = smooth(plane[k], w, h, sigma);
    }
    const std::vector<float>&r = plane[0], &g = plane[1], &bl = plane[2];
    auto diff = [&](int x1, int y1, int x2, int y2) {
        const size_t p = (size_t)y1 * w + x1, q = (size_t)y2 * w + x2;
        const float dr = r[p] - r[q], dg = g[p] - g[q], db = bl[p] - bl[q];
        return std::sqrt(dr * dr + dg * dg + db * db);
    };
    std::vector<Edge> edges;
    edges.reserve(n * 4);
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            const int v = y * w + x;
            if (x < w - 1) edges.push_back(Edge{diff(x, y, x + 1, y), v, v + 1});
            if (y < h - 1) edges.push_back(Edge{diff(x, y, x, y + 1), v, v + w});
            if (x < w - 1 && y < h - 1) edges.push_back(Edge{diff(x, y, x + 1, y + 1), v, v + w + 1});
            if (x < w - 1 && y > 0) edges.push_back(Edge{diff(x, y, x + 1, y - 1), v, v - w + 1});
        }
    Forest u((int)n);
    merge_graph(u, edges, c);
    merge_small(u, edges, min_size);
    return number_components(u, (int)n, labels_out);
}

}  // extern "C"
