// pcm_slic.cuh -- SLIC over-segmentation of the crop on the GPU, the third over-segmentation the reference offers
// (maskers/pixel_classification.py:74-75: slic(crop, n_segments=250, compactness=10, sigma=1, start_label=0)).
//
// The specification is the host code of pcm_slic.cpp, stage by stage; the labels are the same.  Every float64 expression is
// written with __dadd_rn / __dmul_rn / __ddiv_rn in the host code's order, so that nvcc cannot contract it into an FMA:
//   S1 slic_load_kernel     u8 crop -> /255, and the Gaussian's depth pass (axis of length 1)          bit-identical
//   S2 slic_smooth_kernel   Gaussian along rows, then along columns (scipy 'reflect')                  bit-identical
//   S3 slic_lab_kernel      rgb2lab, / compactness                          CUDA's pow / cbrt: <= 1e-12 (DESIGN §10)
//   S4 k-means, max_iter iterations (all run):
//      slic_assign_kernel<false>  one CTA per centre over its +-2 step window: atomicMin of the bit pattern of d
//      slic_assign_kernel<true>   d again; where it equals the minimum, atomicMin of the centre index
//                                 (= the host's "first centre in centre order with the strictly smallest d")
//      slic_settle_kernel         covered pixels take that centre, the others keep the previous iteration's
//      stable radix sort of the pixel indices by centre (CUB), slic_bounds_kernel: each centre's run of pixels
//      slic_update_kernel         one thread per centre sums its pixels in raster order -> means, NaN when empty
//   S5 connectivity enforcement (the host's raster-order capped BFS, in parallel):
//      slic_ccl_*                 4-connected components of the centre map, union-find rooted at the minimum raster index
//      slic_piece_init_kernel     a component of fewer than max_size pixels is one piece
//      slic_split_kernel          larger ones: the host's capped BFS replayed over the component (one thread each)
//      slic_small_kernel          pieces below min_size: BFS replayed, last neighbour in an earlier piece recorded
//      scan of the large pieces -> start_label + rank; slic_jump_kernel resolves the small pieces' chains
//      slic_label_kernel          final labels, n_labels = largest label + 1
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace pcm {

constexpr int SLIC_THREADS = 256;
constexpr int SLIC_NONE = 0x7f7f7f7f;          // "no centre covers this pixel" (byte-fill value of the index pass)

__device__ __forceinline__ int slic_reflect(int i, int n) {     // scipy 'reflect': d c b a | a b c d | d c b a
    while (i < 0 || i >= n) i = i < 0 ? -i - 1 : 2 * n - 1 - i;
    return i;
}

// S1: img = byte / 255 (h*w*3, interleaved as the crop); with `depth`, the Gaussian along the depth axis of length 1:
// a = v*k[r], then a = a + (v+v)*k[r-j] for j = r..1.  Element i of the crop (cx, cy, w, *) of a frame of row stride
// `stride`; the batched Felzenszwalb load runs the same code.
__device__ __forceinline__ double slic_load_value(const uint8_t* __restrict__ frame, long long stride, int cx, int cy, int w,
                                                  const double* __restrict__ k, int radius, int depth, long long i) {
    const long long r = i / (3LL * w), rem = i - r * 3LL * w;
    double v = __ddiv_rn((double)frame[(cy + r) * stride + (long long)cx * 3 + rem], 255.0);
    if (depth) {
        double a = __dmul_rn(v, k[radius]);
        const double vv = __dadd_rn(v, v);
        for (int j = radius; j >= 1; --j) a = __dadd_rn(a, __dmul_rn(vv, k[radius - j]));
        v = a;
    }
    return v;
}

__global__ void __launch_bounds__(SLIC_THREADS) slic_load_kernel(const uint8_t* __restrict__ frame, long long stride, int cx, int cy,
                                                                 int w, int h, const double* __restrict__ k, int radius, int depth,
                                                                 double* __restrict__ out) {
    const long long total = (long long)w * h * 3;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
        out[i] = slic_load_value(frame, stride, cx, cy, w, k, radius, depth, i);
}

// S2: symmetric correlate along one axis (0: rows, 1: columns) of an h x w x 3 image: centre tap first, then the pairs
// from the outside in.  Pixel p of the image; the batched Felzenszwalb smoothing runs the same code.
__device__ __forceinline__ void slic_smooth_pixel(const double* __restrict__ in, double* __restrict__ out, int h, int w, int axis,
                                                  const double* __restrict__ k, int radius, long long p) {
    const int len = axis == 0 ? h : w;
    const long long step = axis == 0 ? 3LL * w : 3;
    const int r = (int)(p / w), c = (int)(p - (long long)r * w);
    const int pos = axis == 0 ? r : c;
    const long long line0 = axis == 0 ? 3LL * c : 3LL * r * w;
    const double* ctr = in + line0 + pos * step;
    const double kc = k[radius];
    double a0 = __dmul_rn(ctr[0], kc), a1 = __dmul_rn(ctr[1], kc), a2 = __dmul_rn(ctr[2], kc);
    for (int j = radius; j >= 1; --j) {
        const double* lo = in + line0 + slic_reflect(pos - j, len) * step;
        const double* hi = in + line0 + slic_reflect(pos + j, len) * step;
        const double wj = k[radius - j];
        a0 = __dadd_rn(a0, __dmul_rn(__dadd_rn(lo[0], hi[0]), wj));
        a1 = __dadd_rn(a1, __dmul_rn(__dadd_rn(lo[1], hi[1]), wj));
        a2 = __dadd_rn(a2, __dmul_rn(__dadd_rn(lo[2], hi[2]), wj));
    }
    double* o = out + 3 * p;
    o[0] = a0; o[1] = a1; o[2] = a2;
}

__global__ void __launch_bounds__(SLIC_THREADS) slic_smooth_kernel(const double* __restrict__ in, double* __restrict__ out, int h, int w,
                                                                   int axis, const double* __restrict__ k, int radius) {
    const long long n = (long long)w * h;
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x)
        slic_smooth_pixel(in, out, h, w, axis, k, radius, p);
}

// S3: rgb2lab of skimage.color on float pixels (channel 0 plays 'R'), times ratio = 1 / compactness.  pow and cbrt are
// CUDA's (not glibc's): the one place where the device may differ from the host, by at most 1e-12 on the output.
__global__ void __launch_bounds__(SLIC_THREADS) slic_lab_kernel(const double* __restrict__ in, double* __restrict__ out, long long n,
                                                                double ratio) {
    const double M[3][3] = {{0.412453, 0.357580, 0.180423}, {0.212671, 0.715160, 0.072169}, {0.019334, 0.119193, 0.950227}};
    const double white[3] = {0.95047, 1.0, 1.08883};
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        double lin[3], f[3];
        for (int c = 0; c < 3; ++c) {
            const double v = in[3 * i + c];
            lin[c] = v > 0.04045 ? pow(__ddiv_rn(__dadd_rn(v, 0.055), 1.055), 2.4) : __ddiv_rn(v, 12.92);
        }
        for (int q = 0; q < 3; ++q) {
            const double t = __ddiv_rn(__dadd_rn(__dadd_rn(__dmul_rn(lin[0], M[q][0]), __dmul_rn(lin[1], M[q][1])), __dmul_rn(lin[2], M[q][2])),
                                       white[q]);
            f[q] = t > 0.008856 ? cbrt(t) : __dadd_rn(__dmul_rn(7.787, t), 16.0 / 116.0);
        }
        out[3 * i + 0] = __dmul_rn(__dsub_rn(__dmul_rn(116.0, f[1]), 16.0), ratio);
        out[3 * i + 1] = __dmul_rn(__dmul_rn(500.0, __dsub_rn(f[0], f[1])), ratio);
        out[3 * i + 2] = __dmul_rn(__dmul_rn(200.0, __dsub_rn(f[1], f[2])), ratio);
    }
}

// S4 assignment, one CTA per centre k over its window (bounds: the host's double expressions and (int) truncation).
//   d = ((0 + ddy) + ddx) * spatial_weight + (((0 + t0^2) + t1^2) + t2^2)   (d >= +0: its bit pattern orders like its value)
// INDEX = false: dmin[o] = min over centres of the bit pattern of d.  INDEX = true: best[o] = smallest k whose d equals it.
template <bool INDEX>
__global__ void __launch_bounds__(SLIC_THREADS) slic_assign_kernel(const double* __restrict__ img, const double* __restrict__ centers,
                                                                   int h, int w, int ty, int tx, double spatial_weight,
                                                                   unsigned long long* __restrict__ dmin, int* __restrict__ best) {
    const int k = blockIdx.x;
    const double* ck = centers + 5LL * k;
    const double cyk = ck[0], cxk = ck[1], c0 = ck[2], c1 = ck[3], c2 = ck[4];
    if (!(cyk == cyk)) return;                                    // a cluster that lost all its pixels
    const int y_min = __double2int_rz(fmax(__dsub_rn(cyk, (double)(2 * ty)), 0.0));
    const int y_max = __double2int_rz(fmin(__dadd_rn(__dadd_rn(cyk, (double)(2 * ty)), 1.0), (double)h));
    const int x_min = __double2int_rz(fmax(__dsub_rn(cxk, (double)(2 * tx)), 0.0));
    const int x_max = __double2int_rz(fmin(__dadd_rn(__dadd_rn(cxk, (double)(2 * tx)), 1.0), (double)w));
    const int ww = x_max - x_min;
    if (ww <= 0 || y_max <= y_min) return;
    const long long total = (long long)(y_max - y_min) * ww;
    for (long long t = threadIdx.x; t < total; t += blockDim.x) {
        const int y = y_min + (int)(t / ww), x = x_min + (int)(t - (t / ww) * ww);
        const double ey = __dsub_rn(cyk, (double)y), ex = __dsub_rn(cxk, (double)x);
        double d = __dmul_rn(__dadd_rn(__dadd_rn(0.0, __dmul_rn(ey, ey)), __dmul_rn(ex, ex)), spatial_weight);
        const long long o = (long long)y * w + x;
        const double* px = img + 3 * o;
        const double t0 = __dsub_rn(px[0], c0), t1 = __dsub_rn(px[1], c1), t2 = __dsub_rn(px[2], c2);
        const double dc = __dadd_rn(__dadd_rn(__dadd_rn(0.0, __dmul_rn(t0, t0)), __dmul_rn(t1, t1)), __dmul_rn(t2, t2));
        d = __dadd_rn(d, dc);
        const unsigned long long bits = (unsigned long long)__double_as_longlong(d);
        if (!INDEX) {
            if (bits < dmin[o]) atomicMin(dmin + o, bits);
        } else if (bits == dmin[o]) {
            atomicMin(best + o, k);
        }
    }
}

__global__ void slic_settle_kernel(const int* __restrict__ best, int* __restrict__ nearest, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        if (best[i] != SLIC_NONE) nearest[i] = best[i];
}

// begin / end of each centre's run in the sorted centre map (runs of empty centres stay 0 / 0)
__global__ void slic_bounds_kernel(const int* __restrict__ keys, int n, int* __restrict__ begin, int* __restrict__ end) {
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const int k = keys[j];
        if (j == 0 || keys[j - 1] != k) begin[k] = j;
        if (j == n - 1 || keys[j + 1] != k) end[k] = j + 1;
    }
}

// S4 update: one thread per centre over its pixels in raster order (the stable sort keeps it), the host's sums
// (0.0 + v_first) + ...; y / x sums are integers and exact.  count 0 -> NaN.
__global__ void slic_update_kernel(const int* __restrict__ sorted_idx, const int* __restrict__ begin, const int* __restrict__ end,
                                   const double* __restrict__ img, int w, int K, double* __restrict__ centers) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    const int b = begin[k], e = end[k];
    long long sy = 0, sx = 0;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0;
    for (int j = b; j < e; ++j) {
        const int p = sorted_idx[j];
        const int y = p / w;
        sy += y;
        sx += p - y * w;
        const double* px = img + 3LL * p;
        s0 = __dadd_rn(s0, px[0]);
        s1 = __dadd_rn(s1, px[1]);
        s2 = __dadd_rn(s2, px[2]);
    }
    double* ck = centers + 5LL * k;
    if (e > b) {
        const double c = (double)(e - b);
        ck[0] = __ddiv_rn((double)sy, c);
        ck[1] = __ddiv_rn((double)sx, c);
        ck[2] = __ddiv_rn(s0, c);
        ck[3] = __ddiv_rn(s1, c);
        ck[4] = __ddiv_rn(s2, c);
    } else {
        const double nan = __longlong_as_double(0x7ff8000000000000LL);
        for (int c = 0; c < 5; ++c) ck[c] = nan;
    }
}

// ---- S5 connectivity ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int slic_find(const int* parent, int x) {
    const volatile int* p = parent;
    int y = p[x];
    while (y != x) { x = y; y = p[x]; }
    return x;
}

// union of the sets of a and b; every parent pointer points to a smaller index, so a root is its set's minimum
__device__ __forceinline__ void slic_unite(int* parent, int a, int b) {
    bool done;
    do {
        a = slic_find(parent, a);
        b = slic_find(parent, b);
        if (a < b) {
            const int old = atomicMin(parent + b, a);
            done = old == b;
            b = old;
        } else if (b < a) {
            const int old = atomicMin(parent + a, b);
            done = old == a;
            a = old;
        } else {
            done = true;
        }
    } while (!done);
}

__global__ void slic_ccl_init_kernel(int* __restrict__ parent, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) parent[i] = i;
}

__global__ void slic_ccl_merge_kernel(const int* __restrict__ seg, int* parent, int w, int h) {
    const int n = w * h;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int y = i / w, x = i - y * w, v = seg[i];
        if (x + 1 < w && seg[i + 1] == v) slic_unite(parent, i, i + 1);
        if (y + 1 < h && seg[i + w] == v) slic_unite(parent, i, i + w);
    }
}

// root[i] = the component's minimum raster index; csize[root] = its pixel count (csize zeroed by the caller)
__global__ void slic_ccl_flatten_kernel(const int* parent, int* __restrict__ root, int* __restrict__ csize, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int r = slic_find(parent, i);
        root[i] = r;
        atomicAdd(csize + r, 1);
    }
}

// a component with fewer than max_size pixels is one piece, started at its root (the host's first BFS there covers it);
// larger ones are left to slic_split_kernel (piece = -1).  psize[start] = size of the piece (zeroed by the caller).
__global__ void slic_piece_init_kernel(const int* __restrict__ root, const int* __restrict__ csize, long long max_size,
                                       int* __restrict__ piece, int* __restrict__ psize, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int r = root[i];
        const int cs = csize[r];
        const bool whole = (long long)cs < max_size;
        piece[i] = whole ? r : -1;
        if (whole && r == i) psize[i] = cs;
    }
}

__constant__ int slic_dy4[4] = {0, 0, 1, -1};
__constant__ int slic_dx4[4] = {1, -1, 0, 0};

// a component of max_size pixels or more: the host's BFS from each not yet assigned pixel in raster order (the component's
// pixels sorted_idx[coff[r] ..], stable-sorted by root), FIFO, neighbours right, left, down, up, stopping as soon as the
// piece has max_size pixels.  One thread per such component; queue[] is the component's own stretch of the scratch.
__global__ void slic_split_kernel(const int* __restrict__ seg, const int* __restrict__ csize, const int* __restrict__ coff,
                                  const int* __restrict__ sorted_idx, int w, int h, long long max_size, int* piece,
                                  int* __restrict__ psize, int* __restrict__ queue) {
    const int n = w * h;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x) {
        const int cs = csize[r];
        if (cs == 0 || (long long)cs < max_size) continue;          // not a root, or a whole-piece component
        const int label = seg[r];
        const int* members = sorted_idx + coff[r];
        int* q = queue + coff[r];
        for (int m = 0; m < cs; ++m) {
            const int s = members[m];
            if (piece[s] >= 0) continue;
            piece[s] = s;
            q[0] = s;
            long long size = 1, visited = 0;
            while (visited < size && size < max_size) {
                const int p = q[visited];
                const int py = p / w, px = p - py * w;
                for (int i = 0; i < 4; ++i) {
                    const int yy = py + slic_dy4[i], xx = px + slic_dx4[i];
                    if (xx >= 0 && xx < w && yy >= 0 && yy < h) {
                        const int o = yy * w + xx;
                        if (seg[o] == label && piece[o] == -1) {
                            piece[o] = s;
                            q[size++] = o;
                            if (size >= max_size) break;
                        }
                    }
                }
                ++visited;
            }
            psize[s] = (int)size;
        }
    }
}

// a piece of fewer than min_size pixels: its BFS replayed in the host's order.  The host keeps the label of the LAST
// neighbour met that lies outside the piece and is already labelled, i.e. belongs to a piece with an earlier start:
// adj[start] = that piece (its final label is resolved later), or -1 for the literal 0.  queue at qoff[start], `seen`
// zeroed by the caller.
__global__ void slic_small_kernel(const int* __restrict__ piece, const int* __restrict__ psize, const int* __restrict__ qoff, int w,
                                  int h, long long min_size, long long max_size, int* __restrict__ queue, int* seen,
                                  int* __restrict__ adj) {
    const int n = w * h;
    for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < n; s += gridDim.x * blockDim.x) {
        const int ps = psize[s];
        if (ps == 0 || (long long)ps >= min_size) continue;
        int* q = queue + qoff[s];
        int adjacent = -1;
        seen[s] = 1;
        q[0] = s;
        long long size = 1, visited = 0;
        while (visited < size && size < max_size) {
            const int p = q[visited];
            const int py = p / w, px = p - py * w;
            for (int i = 0; i < 4; ++i) {
                const int yy = py + slic_dy4[i], xx = px + slic_dx4[i];
                if (xx >= 0 && xx < w && yy >= 0 && yy < h) {
                    const int o = yy * w + xx;
                    const int po = piece[o];
                    if (po == s && !seen[o]) {
                        seen[o] = 1;
                        q[size++] = o;
                        if (size >= max_size) break;
                    } else if (po < s) {
                        adjacent = po;
                    }
                }
            }
            ++visited;
        }
        adj[s] = adjacent;
    }
}

__global__ void slic_flag_kernel(const int* __restrict__ psize, long long min_size, int* __restrict__ flag, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int ps = psize[i];
        flag[i] = ps > 0 && (long long)ps >= min_size;
    }
}

// piece starts: a large piece is its own root with label start_label + rank; a small one points at the piece whose label it
// takes, or is a root with the literal 0
__global__ void slic_link_kernel(const int* __restrict__ psize, const int* __restrict__ rank, const int* __restrict__ adj,
                                 long long min_size, int start_label, int* __restrict__ nxt, int* __restrict__ val, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int ps = psize[i];
        if (ps == 0) continue;
        if ((long long)ps >= min_size) { nxt[i] = i; val[i] = start_label + rank[i]; }
        else if (adj[i] < 0) { nxt[i] = i; val[i] = 0; }
        else nxt[i] = adj[i];
    }
}

// one round of pointer jumping over the piece starts (in place: a pointer only ever moves closer to its root)
__global__ void slic_jump_kernel(const int* __restrict__ psize, int* nxt, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        if (psize[i] > 0) nxt[i] = nxt[nxt[i]];
}

__global__ void slic_label_kernel(const int* __restrict__ piece, const int* __restrict__ nxt, const int* __restrict__ val,
                                  int32_t* __restrict__ labels, int* __restrict__ max_label, int n) {
    int mx = -1;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int v = val[nxt[piece[i]]];
        labels[i] = v;
        mx = max(mx, v);
    }
    for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) atomicMax(max_label, mx);
}

}  // namespace pcm
