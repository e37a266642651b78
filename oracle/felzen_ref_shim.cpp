// felzen_ref_shim.cpp -- TEST INFRASTRUCTURE ONLY.
//
// C-ABI face of the Felzenszwalb-Huttenlocher segmentation the reference vendors under
// prim/src/FelzenSegment (segment-graph.h:48-81 segment_graph, segment_image_index.h:14-121
// segment_image_index).  The reference's headers are #included from where they lie in the
// checkout named by PCM_REFERENCE_ROOT (-I on the compiler command line, see oracle/build_ref.py); nothing of them is
// copied into this repository.  The resulting oracle/_ref/libfelzen_ref.so is used by
// tests/test_felzenszwalb_ref.py to pin the parts of pcm_felzenszwalb that coincide with the
// original algorithm: cost-ordered greedy merge with the k/|C| threshold, union-find, the
// min-size pass.  (scikit-image's variant, which the PC masker actually calls, differs in float
// width, Gaussian and tie order: that part stays "parity unpinned against scikit-image".)
#include <cstring>
#include <vector>

#include "image.h"
#include "misc.h"
#include "filter.h"
#include "segment-graph.h"
#include "segment-image.h"
#include "segment_image_index.h"

extern "C" {

// segment_graph (segment-graph.h:48-81) followed by the min-size pass of segment_image_index.h:85-91
// on a caller-provided edge list.  labels_out[v] = 0-based index of v's component in order of first
// appearance (the numbering of segment_image_index.h:100-113, minus one).  Returns the number of
// components.
int felzen_ref_graph(int n_vertices, int n_edges, const int* a, const int* b, const float* w, float c, int min_size,
                     int* labels_out) {
    std::vector<edge> edges((size_t)n_edges);
    for (int i = 0; i < n_edges; ++i) { edges[i].a = a[i]; edges[i].b = b[i]; edges[i].w = w[i]; }
    universe* u = segment_graph(n_vertices, n_edges, edges.data(), c);
    for (int i = 0; i < n_edges; ++i) {
        int x = u->find(edges[i].a), y = u->find(edges[i].b);
        if ((x != y) && ((u->size(x) < min_size) || (u->size(y) < min_size))) u->join(x, y);
    }
    std::vector<int> index((size_t)n_vertices, -1);
    int next = 0;
    for (int v = 0; v < n_vertices; ++v) {
        int comp = u->find(v);
        if (index[comp] < 0) index[comp] = next++;
        labels_out[v] = index[comp];
    }
    const int n = u->num_sets();
    delete u;
    return n == next ? n : -1;
}

// segment_image_index (segment_image_index.h:14-121) on an h x w x 3 RGB image, row-major u8.
// labels_out[y * w + x] = 0-based component index.  Returns the number of components.
int felzen_ref_image(const unsigned char* rgb_in, int h, int w, float sigma, float c, int min_size, int* labels_out) {
    image<rgb>* im = new image<rgb>(w, h);
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            const unsigned char* p = rgb_in + ((size_t)y * w + x) * 3;
            imRef(im, x, y).r = p[0]; imRef(im, x, y).g = p[1]; imRef(im, x, y).b = p[2];
        }
    int n = 0;
    double* idx = segment_image_index(im, sigma, c, min_size, &n);
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) labels_out[(size_t)y * w + x] = (int)idx[(size_t)x * h + y] - 1;
    delete[] idx;
    delete im;
    return n;
}

}  // extern "C"
