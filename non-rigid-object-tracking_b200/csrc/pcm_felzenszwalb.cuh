// pcm_felzenszwalb.cuh -- Felzenszwalb-Huttenlocher over-segmentation of the crop on the GPU, the second over-segmentation
// the reference offers (maskers/pixel_classification.py:72-73: felzenszwalb(crop, scale=100, sigma=0.5, min_size=50)).
//
// The specification is the host code of pcm_felzenszwalb.cpp; the labels and the count are the same, bit for bit.  Every
// call runs on a chunk of crops (FzCrop; one crop for the single-crop entry points), as one graph of disjoint pieces:
//   F1 fz_load_kernel, two fz_smooth_kernel passes: byte / 255, the Gaussian along rows, then along columns -- the code of
//      slic_load_kernel / slic_smooth_kernel (pcm_slic.cuh), and so the host's smooth_axis, operation for operation
//   F2 fz_cost_kernel      each crop's edges in the host's order (right, down, down-right, up-right; raster order within a
//                          class), crop after crop: endpoints and the bit pattern of sqrt((d0*d0 + d1*d1) + d2*d2)
//   F3 CUB radix sort of (cost bits, edge index): stable, so equal costs keep edge order, as the host's sort does; restricted
//      to one crop it is that crop's own order
//   F4 fz_rounds_kernel<false>   the greedy merge pass, in rounds (below)
//   F5 qs_root_kernel, then fz_rounds_kernel<true>   the min-size pass, in rounds
//   F6 qs_root_kernel + the qs_scan_* kernels (pcm_quickshift.cuh) + fz_label_kernel: label = rank of the root in its crop
// A round decides an edge from its own two components only, and no component spans two crops, so every round makes in
// every crop exactly the decisions that crop makes alone: the labels are the crop's own, and a chunk takes as many rounds
// as its slowest crop.
//
// The merge pass in rounds.  A component X (root = its smallest pixel, as the host's join keeps it) has size[X] and
// limit[X] = Int(X) + sc / |X|.  Each round looks at the remaining edges, in sorted position p, with current roots ra, rb:
//   - ra == rb: dropped (components only grow, so the host finds the same when it reaches the edge);
//   - sA = cost < limit[ra], sB = cost < limit[rb]; m[X] = smallest p of a remaining edge at X whose X side accepts it;
//   - p < m[ra] (or p < m[rb]): every edge at ra up to p fails ra's own limit, so none of them changes ra and the host
//     meets ra as it is now when it reaches p: cost >= limit[ra] rejects the edge whatever happens to rb.  Dropped.
//   - p == m[ra] == m[rb]: by the same argument the host meets both components as they are now, and both sides accept:
//     merged as the host merges (root = smaller index, size = sum, limit = cost + sc / total).  m[X] names one edge per
//     component, so a round's merges form a matching and never touch the same component twice.
//   - every other edge stays for the next round.
// The globally first remaining edge is always decided, so every round makes progress.  An edge keeps the roots of its
// endpoints as of the previous round: after a round of matching merges, parent[old root] is a root again.
// The min-size pass: an edge whose components both have min_size pixels or more is dropped (sizes only grow); any other
// edge the host reaches merges, so one that is the earliest remaining edge of both its components is applied.
// The rounds run in one cooperative kernel with grid-wide syncs, and in its CTA 0 alone once few edges remain: the host
// never waits between rounds.
#pragma once
#include <cooperative_groups.h>
#include <cstdint>
#include <cuda_runtime.h>

#include "pcm_slic.cuh"

namespace pcm {

constexpr int FZ_THREADS = 512;
// once no more edges than this remain, the rounds continue in one CTA: a __syncthreads costs far less than a grid-wide
// sync, and on SegTrack2 crops most rounds see under 1 % of the edges
constexpr int FZ_TAIL_EDGES = 4 * FZ_THREADS;

// One crop of a batched pass.  A chunk of crops is one graph of disjoint pieces: crop k owns the chunk's pixels px ..
// px + w*h - 1 and its edges eb .. eb + edges(w, h) - 1, in crop order; its labels go to `labels` (w*h, raster order).
struct FzCrop {
    const uint8_t* frame;          // the frame the crop is cut from (row stride: the batch's)
    int32_t* labels;
    int cx, cy, w, h;
    int px, eb;                    // pixel base and edge base within the chunk
};

__host__ __device__ __forceinline__ long long fz_edge_count(int w, int h) {
    return (long long)h * (w - 1) + (long long)(h - 1) * w + 2LL * (h - 1) * (w - 1);
}

// the crop of chunk element v: the last of the n crops whose pixel base (EDGE = false) or edge base (true) is <= v (a
// crop without edges shares its edge base with the next one)
template <bool EDGE>
__device__ __forceinline__ int fz_crop_of(const FzCrop* __restrict__ crops, int n, long long v) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((EDGE ? crops[mid].eb : crops[mid].px) <= v) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// F1 of a chunk: pixel-channel i -> byte / 255 (slic_load_value, depth 0) into img, the chunk's pixels back to back
__global__ void __launch_bounds__(256) fz_load_kernel(const FzCrop* __restrict__ crops, int n_crops, long long stride, int n_px,
                                                      double* __restrict__ img) {
    const long long total = 3LL * n_px;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const FzCrop c = crops[fz_crop_of<false>(crops, n_crops, i / 3)];
        img[i] = slic_load_value(c.frame, stride, c.cx, c.cy, c.w, nullptr, 0, 0, i - 3LL * c.px);
    }
}

// F1 of a chunk: the Gaussian along rows (axis 0) or columns (1) of every crop (slic_smooth_pixel)
__global__ void __launch_bounds__(256) fz_smooth_kernel(const FzCrop* __restrict__ crops, int n_crops, int n_px,
                                                        const double* __restrict__ in, double* __restrict__ out, int axis,
                                                        const double* __restrict__ k, int radius) {
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n_px; p += gridDim.x * blockDim.x) {
        const FzCrop c = crops[fz_crop_of<false>(crops, n_crops, p)];
        slic_smooth_pixel(in + 3LL * c.px, out + 3LL * c.px, c.h, c.w, axis, k, radius, p - c.px);
    }
}

// F2: edge i of the host's array for an h x w image: endpoints (a, b) and the bit pattern of its cost (>= +0, so the bits
// order like the value)
__device__ __forceinline__ unsigned long long fz_edge(const double* __restrict__ img, int h, int w, long long i, int& a, int& b) {
    const long long n_right = (long long)h * (w - 1), n_down = (long long)(h - 1) * w, n_diag = (long long)(h - 1) * (w - 1);
    if (i < n_right) {                                      // (r, c) - (r, c-1), c >= 1
        const int r = (int)(i / (w - 1)), c = (int)(i - (long long)r * (w - 1)) + 1;
        a = r * w + c; b = a - 1;
    } else if (i < n_right + n_down) {                      // (r, c) - (r-1, c), r >= 1
        const long long j = i - n_right;
        a = (int)j + w; b = (int)j;
    } else {
        const long long j = i - n_right - n_down;
        const bool dr = j < n_diag;                         // down-right: (r, c) - (r-1, c-1); up-right: (r-1, c) - (r, c-1)
        const long long k = dr ? j : j - n_diag;
        const int r = (int)(k / (w - 1)) + 1, c = (int)(k - (long long)(r - 1) * (w - 1)) + 1;
        if (dr) { a = r * w + c; b = (r - 1) * w + c - 1; }
        else    { a = (r - 1) * w + c; b = r * w + c - 1; }
    }
    const double* p = img + 3LL * a;
    const double* q = img + 3LL * b;
    const double d0 = __dsub_rn(p[0], q[0]), d1 = __dsub_rn(p[1], q[1]), d2 = __dsub_rn(p[2], q[2]);
    const double c = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(d0, d0), __dmul_rn(d1, d1)), __dmul_rn(d2, d2)));
    return (unsigned long long)__double_as_longlong(c);
}

// F2 of a chunk: edge i = edge i - eb of its crop, endpoints as chunk pixel indices; idx = i, so that the stable sort
// keeps crop k's edges after crop k-1's and, within a crop, in the host's order
__global__ void __launch_bounds__(256) fz_cost_kernel(const FzCrop* __restrict__ crops, int n_crops, int n_edges,
                                                      const double* __restrict__ img, int* __restrict__ ea, int* __restrict__ eb,
                                                      unsigned long long* __restrict__ key, int* __restrict__ idx) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_edges; i += gridDim.x * blockDim.x) {
        const FzCrop c = crops[fz_crop_of<true>(crops, n_crops, i)];
        int a, b;
        key[i] = fz_edge(img + 3LL * c.px, c.h, c.w, i - c.eb, a, b);
        ea[i] = c.px + a;
        eb[i] = c.px + b;
        idx[i] = i;
    }
}

// The edge list the rounds work on: sorted position p and the current roots of the endpoints (p = -1: dropped this round)
struct alignas(16) FzEdge { int p, a, b, pad; };

// every pixel its own component: parent = i, size = 1, limit = 0.0 + sc / 1 (limit0, computed by the host as its code does)
__global__ void __launch_bounds__(256) fz_init_kernel(int* __restrict__ parent, int* __restrict__ size, double* __restrict__ limit,
                                                      double limit0, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        parent[i] = i;
        size[i] = 1;
        limit[i] = limit0;
    }
}

// list[p] = edge at sorted position p with endpoints root[a], root[b] (root == nullptr: the pixels themselves); the
// counters of fz_rounds_kernel set for this list
__global__ void __launch_bounds__(256) fz_gather_kernel(const int* __restrict__ sorted_idx, const int* __restrict__ ea,
                                                        const int* __restrict__ eb, const int* __restrict__ root, int n_edges,
                                                        FzEdge* __restrict__ list, int* __restrict__ ctr) {
    if (blockIdx.x == 0 && threadIdx.x < 4) ctr[threadIdx.x] = threadIdx.x == 0 ? n_edges : 0;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n_edges; p += gridDim.x * blockDim.x) {
        const int e = sorted_idx[p];
        int a = ea[e], b = eb[e];
        if (root) { a = root[a]; b = root[b]; }
        list[p] = {p, a, b, 0};
    }
}

struct FzRounds {
    int* parent;                   // parent pointers, towards the smaller index
    int* size;
    double* limit;                 // merge pass: Int(X) + sc / |X| of each root
    unsigned long long* m;         // per root: (~round << 32) | earliest position; entries of other rounds read as "none"
    const unsigned long long* key; // sorted cost bits, by position
    FzEdge* list[2];               // the remaining edges of even / odd rounds
    int* ctr;                      // [0..1] list sizes, [2..3] edges that survive the first filter of a round
    int* rounds;                   // the number of rounds taken
    double sc;
    int min_size;
};

// the rounds read what other CTAs wrote in earlier rounds: loads bypass L1
__device__ __forceinline__ FzEdge fz_load(const FzEdge* e) {
    const int4 v = __ldcg(reinterpret_cast<const int4*>(e));
    return {v.x, v.y, v.z, v.w};
}
__device__ __forceinline__ unsigned long long fz_stamp(int round, int p) {
    return ((unsigned long long)(0xffffffffu - (unsigned)round) << 32) | (unsigned)p;
}
__device__ __forceinline__ int fz_earliest(const unsigned long long* m, int x, int round) {
    const unsigned long long v = __ldcg(m + x);
    return (unsigned)(v >> 32) == 0xffffffffu - (unsigned)round ? (int)(unsigned)v : 0x7fffffff;
}

// Rounds of the merge pass (MIN_SIZE = false) or of the min-size pass (true) until no edge remains; ctr[0] holds the size
// of the initial list (list[0]), ctr[1..3] are 0.  Launched cooperatively: every block is resident.
template <bool MIN_SIZE>
__global__ void __launch_bounds__(FZ_THREADS, 1) fz_rounds_kernel(FzRounds s) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ int block_count;
    const int lane = threadIdx.x & 31;
    volatile int* ctr = s.ctr;
    int round = 0;
    bool single = false;                                        // the tail: CTA 0 alone
    for (;;) {
        ++round;
        const int cur = (round - 1) & 1, nxt = round & 1;
        const int n = ctr[cur];
        if (!single && n <= FZ_TAIL_EDGES) {                    // every CTA reads the same n
            if (blockIdx.x != 0) return;
            single = true;
        }
        const int tid = (single ? 0 : blockIdx.x) * FZ_THREADS + threadIdx.x;
        const int stride = (single ? 1 : gridDim.x) * FZ_THREADS;
        FzEdge* in = cur ? s.list[1] : s.list[0];             // (no dynamic index into the parameter: no local copy)
        FzEdge* out = cur ? s.list[0] : s.list[1];
        if (tid == 0) { ctr[nxt] = 0; ctr[2 + nxt] = 0; }      // read for the last time in the previous round
        if (threadIdx.x == 0) block_count = 0;
        __syncthreads();
        // first filter: current roots, drop edges inside one component (and, in the min-size pass, between two large ones),
        // record each component's earliest position
        int kept = 0;
        for (int i = tid; i < n; i += stride) {
            FzEdge e = fz_load(in + i);
            const int ra = __ldcg(s.parent + e.a), rb = __ldcg(s.parent + e.b);
            bool live = ra != rb;
            if (MIN_SIZE && live) live = __ldcg(s.size + ra) < s.min_size || __ldcg(s.size + rb) < s.min_size;
            if (!live) {
                e.p = -1;
            } else {
                ++kept;
                const unsigned long long st = fz_stamp(round, e.p);
                if (MIN_SIZE) {
                    atomicMin(s.m + ra, st);
                    atomicMin(s.m + rb, st);
                } else {
                    const double c = __longlong_as_double((long long)s.key[e.p]);
                    if (c < __ldcg(s.limit + ra)) atomicMin(s.m + ra, st);
                    if (c < __ldcg(s.limit + rb)) atomicMin(s.m + rb, st);
                }
                e.a = ra;
                e.b = rb;
            }
            in[i] = e;
        }
        for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
        if (lane == 0 && kept) atomicAdd(&block_count, kept);
        __syncthreads();
        if (threadIdx.x == 0 && block_count) atomicAdd((int*)ctr + 2 + cur, block_count);
        if (single) __syncthreads(); else grid.sync();
        if (ctr[2 + cur] == 0) break;
        // second filter: certain rejections go, certain merges are applied, the rest is kept for the next round
        for (int base = tid - (int)threadIdx.x; base < n; base += stride) {
            const int i = base + threadIdx.x;
            bool keep = false;
            if (i < n) {
                const FzEdge e = fz_load(in + i);
                if (e.p >= 0) {
                    const int ma = fz_earliest(s.m, e.a, round), mb = fz_earliest(s.m, e.b, round);
                    if (e.p == ma && e.p == mb) {
                        const int r = min(e.a, e.b), o = max(e.a, e.b);
                        const int total = __ldcg(s.size + e.a) + __ldcg(s.size + e.b);
                        s.parent[o] = r;
                        s.size[r] = total;
                        if (!MIN_SIZE)
                            s.limit[r] = __dadd_rn(__longlong_as_double((long long)s.key[e.p]), __ddiv_rn(s.sc, (double)total));
                    } else {
                        keep = MIN_SIZE || (e.p >= ma && e.p >= mb);
                    }
                }
            }
            const unsigned ballot = __ballot_sync(0xffffffffu, keep);
            if (ballot) {
                int at = 0;
                if (lane == 0) at = atomicAdd((int*)ctr + nxt, __popc(ballot));
                at = __shfl_sync(0xffffffffu, at, 0);
                if (keep) out[at + __popc(ballot & ((1u << lane) - 1))] = fz_load(in + i);
            }
        }
        if (single) __syncthreads(); else grid.sync();
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *s.rounds = round - 1;
}

// F6 of a chunk: roots are the smallest chunk pixel of their component, so within a crop they come in the crop's raster
// order.  rank = exclusive scan of the root flags over the chunk, total = number of roots: crop k's label of pixel p is
// rank[root[p]] - rank[px], its count rank[next crop's px] (or total) - rank[px], written by the crop's first pixel.
__global__ void __launch_bounds__(256) fz_label_kernel(const FzCrop* __restrict__ crops, int n_crops, int n_px,
                                                       const int* __restrict__ root, const int* __restrict__ rank,
                                                       const int* __restrict__ total, int* __restrict__ counts) {
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n_px; p += gridDim.x * blockDim.x) {
        const int k = fz_crop_of<false>(crops, n_crops, p);
        const FzCrop c = crops[k];
        const int base = rank[c.px];
        c.labels[p - c.px] = rank[root[p]] - base;
        if (p == c.px) counts[k] = (k + 1 < n_crops ? rank[crops[k + 1].px] : *total) - base;
    }
}

}  // namespace pcm
