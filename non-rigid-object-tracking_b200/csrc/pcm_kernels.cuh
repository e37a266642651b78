// pcm_kernels.cuh -- CUDA kernels of the PC masker hot path (sm_100a).
//
//  K0 planes_kernel, K1 score_kernel: pcm_score.cuh
//  Kn novelty_kernel      PCA reconstruction error of models with two or more components, between K0 and K1
//  K2 segment_decide      per-label score and decision (:240-242); labels inside the guard
//                         band are re-evaluated exactly (sequential float32, raster order) from
//                         per-pixel values the block recomputes for the label's bounding box
//  K3 mask_dilate         decision -> 0/255 map (:242-246) fused with cv.dilate (:112)
//  K5 iou_kernel          computeBenchmark counts (benchmark.py:8-14)
//  + convert_kernel / gather_kernel: parity taps (pcm_convert, pcm_gather_features)
#pragma once
#include "pcm_score.cuh"

namespace pcm {

// Kn -----------------------------------------------------------------------------
// Novelty error of PCAs with two or more components (params.n_components > 1; :57-63, :88-93 with
// PCA(n_components=k), :203-213).  Launched between K0 and K1 for a frame whose current or next model has such a PCA;
// it writes the blended error of every crop pixel (blend2, as K1 blends), and K1 and K2's exact path read that map
// instead of computing the term themselves, so both use the same bits.  Rank-1 models keep K1's in-line pass
// (novelty_error, pcm_score.cuh) unless blended with a higher-rank one.
//
// Arithmetic (scikit-learn's transform / inverse_transform, whiten=False), per pixel and model, with x_f = v_f / 255
// (v_f the plane byte, -1 outside the crop):
//   t_j  = S_j / 255 - mdc_j,   S_j = sum_f v_f c_jf accumulated with fma (exact v_f),   mdc_j = mean . c_j (host,
//          feature order)                                                        -> t_j = x . c_j - mean . c_j
//   r_f  = fma(t_{k-1}, c_{k-1,f}, ... fma(t_1, c_1f, fma(t_0, c_0f, mean_f)))      -> mean_f + sum_j t_j c_jf
//   err  = sum_f |fma(v_f, 1/255, -r_f)|                                             -> sum_f |x_f - r_f|
// Every sum runs over the features in K1's order: tap by tap, plane by plane (entry it = k * nch + p holds feature
// (p / 3) * 3K + 3k + p % 3).  The coefficients of a model are laid out in that order, k + 1 doubles per entry
// ({c_0f .. c_{k-1}f, mean_f}), and staged in shared memory when they fit (always on sm_100: two models of F <= 1161,
// k <= 8 take 167 KB), else read through L1.
// A CTA scores tiles of NOV_TW x NOV_TH pixels (persistent, grid-stride); a thread owns NOV_PIX consecutive rows of one
// column, so every coefficient load serves NOV_PIX pixels.  Plane bytes are read through L1 (the 2n+1 rows of taps of
// a tile are reused by all of its pixels).
constexpr int MAX_PCA_K = 8;
constexpr int NOV_PIX = 4, NOV_TW = 32, NOV_TH = (NTHREADS / 32) * NOV_PIX;

struct NoveltyArgs {
    const uint8_t* planes;     // K0's planar crop (as PixelScorer)
    long long pitch, plane_stride;
    int cw, ch;
    int row0, rows;            // crop rows [row0, row0 + rows) of this launch
    Geom g;
    const double* coef0;       // model 0: [F][k0 + 1] in visiting order (see above)
    const double* coef1;       // model 1 (blend)
    int k0, k1;
    double mdc0[MAX_PCA_K], mdc1[MAX_PCA_K];
    int blend;
    double w0, w1;
    int staged;                // 1: coefficients copied to shared memory
    double* out;               // [ch*cw]
};

__host__ __device__ inline size_t novelty_smem_bytes(const Geom& g, int k0, int k1, bool blend, bool staged) {
    return staged ? sizeof(double) * (size_t)g.F * ((k0 + 1) + (blend ? k1 + 1 : 0)) : 0;
}

template <int KC>
__device__ __forceinline__ void pca_l1_error(const NoveltyArgs& a, const double* coef, const double* mdc,
                                             int x, int y, double (&err)[NOV_PIX]) {
    const Geom& g = a.g;
    const int nch = 3 * g.n_spaces;
    double t[KC][NOV_PIX];
#pragma unroll
    for (int i = 0; i < NOV_PIX; ++i) {
        err[i] = 0.0;
#pragma unroll
        for (int j = 0; j < KC; ++j) t[j][i] = 0.0;
    }
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
        const double* c = coef;
#pragma unroll 1
        for (int k = 0; k < g.K; ++k) {
            int dr, dc;
            star_tap(k, dr, dc);
            const int xx = x + dc;
            long long off[NOV_PIX];
            bool ok[NOV_PIX];
#pragma unroll
            for (int i = 0; i < NOV_PIX; ++i) {
                const int yy = y + i + dr;
                ok[i] = xx >= 0 && xx < a.cw && yy >= 0 && yy < a.ch;
                off[i] = ok[i] ? (long long)yy * a.pitch + xx : 0;
            }
#pragma unroll 1
            for (int p = 0; p < nch; ++p, c += KC + 1) {
                const uint8_t* plane = a.planes + (long long)p * a.plane_stride;
                double xv[NOV_PIX];   // v_f
#pragma unroll
                for (int i = 0; i < NOV_PIX; ++i) xv[i] = ok[i] ? u8_to_double(__ldg(plane + off[i])) : -1.0;
                if (pass == 0) {
#pragma unroll
                    for (int j = 0; j < KC; ++j) {
                        const double cj = c[j];
#pragma unroll
                        for (int i = 0; i < NOV_PIX; ++i) t[j][i] = fma(xv[i], cj, t[j][i]);
                    }
                } else {
                    double r[NOV_PIX];
                    const double mu = c[KC];
#pragma unroll
                    for (int i = 0; i < NOV_PIX; ++i) r[i] = mu;
#pragma unroll
                    for (int j = 0; j < KC; ++j) {
                        const double cj = c[j];
#pragma unroll
                        for (int i = 0; i < NOV_PIX; ++i) r[i] = fma(t[j][i], cj, r[i]);
                    }
#pragma unroll
                    for (int i = 0; i < NOV_PIX; ++i) err[i] += fabs(fma(xv[i], 1.0 / 255.0, -r[i]));
                }
            }
        }
        if (pass == 0) {
#pragma unroll
            for (int j = 0; j < KC; ++j)
#pragma unroll
                for (int i = 0; i < NOV_PIX; ++i) t[j][i] = __dsub_rn(__ddiv_rn(t[j][i], 255.0), mdc[j]);
        }
    }
}

__device__ __forceinline__ void pca_l1_error_k(int k, const NoveltyArgs& a, const double* coef, const double* mdc,
                                               int x, int y, double (&err)[NOV_PIX]) {
    switch (k) {
        case 1: pca_l1_error<1>(a, coef, mdc, x, y, err); break;
        case 2: pca_l1_error<2>(a, coef, mdc, x, y, err); break;
        case 3: pca_l1_error<3>(a, coef, mdc, x, y, err); break;
        case 4: pca_l1_error<4>(a, coef, mdc, x, y, err); break;
        case 5: pca_l1_error<5>(a, coef, mdc, x, y, err); break;
        case 6: pca_l1_error<6>(a, coef, mdc, x, y, err); break;
        case 7: pca_l1_error<7>(a, coef, mdc, x, y, err); break;
        default: pca_l1_error<8>(a, coef, mdc, x, y, err); break;
    }
}

__global__ void __launch_bounds__(NTHREADS) novelty_kernel(const NoveltyArgs a) {
    extern __shared__ __align__(16) double nsm[];
    const double* c0 = a.coef0;
    const double* c1 = a.coef1;
    if (a.staged) {                                       // model state only: overlaps K0's tail under PDL
        const int n0 = (a.k0 + 1) * a.g.F, n1 = a.blend ? (a.k1 + 1) * a.g.F : 0;
        double* s0 = nsm;
        double* s1 = s0 + n0;
        for (int i = threadIdx.x; i < n0; i += blockDim.x) s0[i] = a.coef0[i];
        for (int i = threadIdx.x; i < n1; i += blockDim.x) s1[i] = a.coef1[i];
        c0 = s0;
        c1 = s1;
    }
    grid_dependency_wait();     // K0's planes are complete and visible (and, since K0 waits too, everything before K0)
    grid_launch_dependents();
    __syncthreads();
    const int tiles_x = (a.cw + NOV_TW - 1) / NOV_TW, tiles_y = (a.rows + NOV_TH - 1) / NOV_TH;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int tile = blockIdx.x; tile < tiles_x * tiles_y; tile += gridDim.x) {
        const int x = (tile % tiles_x) * NOV_TW + lane;
        const int y = a.row0 + (tile / tiles_x) * NOV_TH + warp * NOV_PIX;
        double e[NOV_PIX];
        pca_l1_error_k(a.k0, a, c0, a.mdc0, x, y, e);
        if (a.blend) {
            double e1[NOV_PIX];
            pca_l1_error_k(a.k1, a, c1, a.mdc1, x, y, e1);
#pragma unroll
            for (int i = 0; i < NOV_PIX; ++i) e[i] = blend2(e[i], e1[i], a.w0, a.w1);
        }
        if (x < a.cw) {
#pragma unroll
            for (int i = 0; i < NOV_PIX; ++i)
                if (y + i < a.row0 + a.rows) a.out[(size_t)(y + i) * a.cw + x] = e[i];
        }
    }
}

// K2 -----------------------------------------------------------------------------
// score = f32( (acc/area) * (1-w) + prior * w ) > 0.5 (:241-242), acc being the
// reference's sequential float32 accumulator.  Every one of its `area` adds rounds a partial sum of
// magnitude <= sum|d| to float32 (relative error 2^-24), so acc differs from the exact sum by at most
// area * 2^-24 * sum|d| and the score by 2^-24 * sum|d| * |1-w|; a label whose score is that close to
// 0.5 (plus the roundings of the score expression itself) is re-evaluated EXACTLY by its block: float32 accumulator, each
// `+=` evaluated in float64 and rounded to float32, pixels in raster order (:235-238).
//
// The per-pixel values d of such a label are not stored by K1 (that would be 8 - 16 bytes per pixel of every frame for
// the sake of about one label in ten frames): the block recomputes them for the pixels of the label's bounding box from
// the colour planes in global memory -- same nodes, same leaf values, same operations in the same order as K1
// (ps_forest / ps_novelty below), so the values are bit-identical.  With pcm_set_debug the maps ARE stored and read back.
struct PixelScorer {
    const uint8_t* planes;     // K0's planar crop: plane p at planes + p * plane_stride, rows `pitch` apart
    long long pitch, plane_stride;
    int cw, ch;
    Geom g;
    DevForest f0, f1;
    int depth, blend;
    double w0, w1;
    int novelty;               // rank-1 novelty term, recomputed by ps_novelty
    DevPCA pca0, pca1;
    const double* nov_map;     // [ch*cw] novelty_kernel's blended error (PCAs of rank >= 2), or nullptr
};

// the tile byte offset a node carries -> the plane sample of pixel (x, y) it means (0 outside the crop, like the TMA fill)
__device__ __forceinline__ unsigned ps_sample(const PixelScorer& s, int x, int y, unsigned tap) {
    const unsigned plane = tap / (unsigned)s.g.PS, rem = tap - plane * (unsigned)s.g.PS;
    const int r = y + (int)(rem / (unsigned)s.g.RS) - s.g.n, c = x + (int)(rem % (unsigned)s.g.RS) - s.g.HX;
    if (r < 0 || r >= s.ch || c < 0 || c >= s.cw) return 0u;
    return __ldg(s.planes + (long long)plane * s.plane_stride + (long long)r * s.pitch + c);
}

// mean leaf fraction of one forest, trees added in estimator order (four walked at a time for latency)
__device__ double ps_forest(const PixelScorer& s, const DevForest& f, int x, int y) {
    const uint8_t* nodes = reinterpret_cast<const uint8_t*>(f.nodes);
    const uint8_t* leaves = reinterpret_cast<const uint8_t*>(f.leaves);
    double acc = 0.0;
    for (int t0 = 0; t0 < f.n_trees; t0 += 4) {
        unsigned ref[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) ref[q] = (unsigned)f.trees[min(t0 + q, f.n_trees - 1)].x;
        for (int l = 0; l < s.depth; ++l) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const NodeT nd = __ldg(reinterpret_cast<const NodeT*>(nodes + ref[q]));
                const unsigned v = ps_sample(s, x, y, node_tap(nd));
                ref[q] = node_left(nd) + (v > node_thr(nd) ? NODE_BYTES : 0u);
            }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (t0 + q < f.n_trees) acc = __dadd_rn(acc, __ldg(reinterpret_cast<const double*>(leaves + ref[q])));
    }
    return __ddiv_rn(acc, (double)f.n_trees);
}

// novelty_error of pcm_score.cuh for one pixel: features tap by tap, plane by plane
__device__ double ps_novelty(const PixelScorer& s, const DevPCA& pca, int x, int y) {
    const Geom& g = s.g;
    const int nch = 3 * g.n_spaces;
    double t = 0.0, err = 0.0;
    for (int pass = 0; pass < 2; ++pass) {
        for (int k = 0; k < g.K; ++k) {
            int dr, dc;
            star_tap(k, dr, dc);
            const unsigned off = (unsigned)((dr + g.n) * g.RS + (dc + g.HX));
            const bool ok = ps_sample(s, x, y, (unsigned)(nch * g.PS) + off) != 0;
            for (int p = 0; p < nch; ++p) {
                const int f = (p / 3) * 3 * g.K + 3 * k + (p % 3);
                const double v = ok ? u8_to_double(ps_sample(s, x, y, (unsigned)(p * g.PS) + off)) : -1.0;
                if (pass == 0) t = fma(v, pca.comp255[f], t);
                else err += fabs(fma(v, 1.0 / 255.0, -fma(t, pca.comp[f], pca.mean[f])));
            }
        }
        if (pass == 0) t -= pca.mean_dot_comp;
    }
    return err;
}

__device__ double ps_contribution(const PixelScorer& s, int x, int y, double thr) {
    double p = ps_forest(s, s.f0, x, y);
    if (s.blend) p = blend2(p, ps_forest(s, s.f1, x, y), s.w0, s.w1);
    double e = 0.0;
    if (s.nov_map) {
        e = s.nov_map[(size_t)y * s.cw + x];        // the value K1 read: identical bits
    } else if (s.novelty) {
        e = ps_novelty(s, s.pca0, x, y);
        if (s.blend) e = blend2(e, ps_novelty(s, s.pca1, x, y), s.w0, s.w1);
    }
    return contribution(p, e, thr);
}

struct DecideArgs {
    const double* p1;          // per-pixel maps kept by K1 (pcm_set_debug), or nullptr: recompute (ps)
    const double* sa;          // nullptr when novelty is off or the maps are not kept
    PixelScorer ps;
    const int32_t* labels;
    int cw;
    double thr;
    const double* sum;
    const double* asum;
    const int* area;
    const int* rmin;
    const int* rmax;
    const int* cmin;
    const int* cmax;
    const float* priors;       // nullptr -> all -1
    int n_labels;
    double prior_weight;
    uint8_t* decision;         // [S] 0/1
    float* scores;             // [S]
    int* n_flagged;            // number of labels that took the exact path
    int force_exact;           // test hook (pcm_set_debug bit 1): every label takes the exact path
};

__global__ void __launch_bounds__(256) segment_decide_kernel(const DecideArgs a) {
    __shared__ int s_list[256];
    __shared__ int s_n;
    __shared__ double s_d[256];
    __shared__ unsigned char s_m[256];
    grid_dependency_wait();
    grid_launch_dependents();
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const double w = a.prior_weight;
    const double omw = __dsub_rn(1.0, w);
    if (s < a.n_labels) {
        // independent loads first: this kernel is one dependent-latency chain per label otherwise
        const int area = a.area[s];
        const double sum = a.sum[s], asum = a.asum[s];
        const double prior = a.priors ? (double)a.priors[s] : -1.0;
        if (area <= 0) { a.decision[s] = 0; a.scores[s] = 0.f; }
        else {
            const double sc = __dadd_rn(__dmul_rn(__ddiv_rn(sum, (double)area), omw), __dmul_rn(prior, w));
            const double band = 5.9604644775390625e-08 * asum * fabs(omw) * 1.0000001 + 2.4e-7;
            a.decision[s] = sc > 0.5;
            a.scores[s] = (float)sc;
            if (a.force_exact || fabs(sc - 0.5) <= band) s_list[atomicAdd(&s_n, 1)] = s;
        }
    }
    __syncthreads();
    const int n_flagged = s_n;
    if (n_flagged == 0) return;
    if (threadIdx.x == 0) atomicAdd(a.n_flagged, n_flagged);
    for (int f = 0; f < n_flagged; ++f) {
        const int L = s_list[f];
        const int r0 = a.rmin[L], r1 = a.rmax[L], c0 = a.cmin[L], c1 = a.cmax[L];
        const int bw = c1 - c0 + 1, npos = bw * (r1 - r0 + 1);
        float acc = 0.f;                                   // thread 0: the reference's float32 accumulator
        for (int base = 0; base < npos; base += 256) {
            const int q = base + threadIdx.x;
            bool mine = false;
            double d = 0.0;
            if (q < npos) {
                const int r = r0 + q / bw, c = c0 + q % bw;
                const int idx = r * a.cw + c;
                mine = a.labels[idx] == L;
                if (mine) d = a.p1 ? contribution(a.p1[idx], a.sa ? a.sa[idx] : 0.0, a.thr) : ps_contribution(a.ps, c, r, a.thr);
            }
            s_m[threadIdx.x] = mine;
            s_d[threadIdx.x] = d;
            __syncthreads();
            if (threadIdx.x == 0) {
                const int n = min(256, npos - base);
                for (int i = 0; i < n; ++i)                // raster order inside the bounding box = raster order of the crop
                    if (s_m[i]) acc = __double2float_rn(__dadd_rn((double)acc, s_d[i]));
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            const double prior = a.priors ? (double)a.priors[L] : -1.0;
            const float sc = __double2float_rn(__dadd_rn(__dmul_rn(__ddiv_rn((double)acc, (double)a.area[L]), omw),
                                                         __dmul_rn(prior, w)));
            a.scores[L] = sc;
            a.decision[L] = sc > 0.5f;
        }
    }
}

// K3 -----------------------------------------------------------------------------
// map[r][c] = 255 * decision[label[r][c]] (:242-245) followed by cv.dilate with a
// k x k box, anchor (k/2, k/2), neighbours outside the crop ignored (:112).
struct DilateArgs {
    const int32_t* labels;
    const uint8_t* decision;
    int cw, ch, k, n_labels;
    uint8_t* mask;             // dense plane; element (cy + r, cx + c)
    long long mask_stride;
    int cx, cy;
    uint8_t* pre;              // optional [ch*cw] pre-dilation map
};

constexpr int DIL_TW = 128, DIL_TH = 32, DIL_MAXK = 33;
constexpr int DIL_SH_MAX = DIL_TH + DIL_MAXK - 1;                 // staged rows incl. halo
constexpr int DIL_PITCH = DIL_TW + 4 * ((DIL_MAXK + 2) / 4 + 1);   // staged row pitch (bytes, multiple of 4)
static_assert(DIL_MAXK - 1 <= 32, "one halo label per lane");

// One block = 128 x 32 output pixels, 8 warps.
//   stage 1  decision[label] for the tile plus its k-1 halo -> s0 (0/1 bytes).  A warp owns whole
//            rows: each lane fetches four labels of the tile interior with one 16-byte load (when
//            the label rows are 16-byte aligned) and lanes < k-1 fetch one halo label; the loads
//            of a batch of rows are all in flight before the dependent decision loads.  The
//            interior starts at a 4-byte aligned column of s0 (PAD bytes of left padding).
//   stage 2  OR along rows, four pixels per thread: the k shifted windows of a 32-bit word come
//            from funnel shifts of adjacent words (SWAR) -> s1
//   stage 3  OR along columns on 32-bit words, * 255, one 4-byte store per thread
// KF > 0: kernel size fixed at compile time (7 = every config of the reference); KF = 0: a.k
template <bool VEC, bool PRE, int KF>
__global__ void __launch_bounds__(256) mask_dilate_kernel(const DilateArgs a) {
    __shared__ __align__(16) uint8_t s0[DIL_SH_MAX * DIL_PITCH];
    __shared__ __align__(16) uint8_t s1[DIL_SH_MAX * DIL_TW];
    grid_dependency_wait();
    grid_launch_dependents();
    const int k = KF > 0 ? KF : a.k, before = k / 2, after = k - 1 - before, SH = DIL_TH + k - 1;
    const int pad = (4 - (before & 3)) & 3;         // s0 column of tile column x is x - tx0 + before + pad
    const int tx0 = blockIdx.x * DIL_TW, ty0 = blockIdx.y * DIL_TH;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x4 = tx0 + 4 * lane;                  // first of the lane's four interior columns
    // halo column of this lane: lanes [0, before) left of the tile, [before, k-1) right of it
    const int hx = lane < before ? tx0 - before + lane : tx0 + DIL_TW + (lane - before);
    const bool h_on = lane < k - 1 && hx >= 0 && hx < a.cw;
    const int hs = hx - tx0 + before + pad;         // its s0 column
    constexpr int RB = 4;                           // rows per batch of a warp
    for (int r0 = warp * RB; r0 < SH; r0 += 8 * RB) {
        int4 v4[RB];
        int vh[RB];
#pragma unroll
        for (int q = 0; q < RB; ++q) {
            const int r = r0 + q, y = ty0 - before + r;
            const bool row_ok = r < SH && y >= 0 && y < a.ch;
            const int32_t* lrow = a.labels + (size_t)(row_ok ? y : 0) * a.cw;
            v4[q] = make_int4(-1, -1, -1, -1);
            if (row_ok) {
                if (VEC && x4 + 3 < a.cw) v4[q] = __ldg(reinterpret_cast<const int4*>(lrow + x4));
                else {
                    if (x4 + 0 < a.cw) v4[q].x = __ldg(lrow + x4 + 0);
                    if (x4 + 1 < a.cw) v4[q].y = __ldg(lrow + x4 + 1);
                    if (x4 + 2 < a.cw) v4[q].z = __ldg(lrow + x4 + 2);
                    if (x4 + 3 < a.cw) v4[q].w = __ldg(lrow + x4 + 3);
                }
            }
            vh[q] = (row_ok && h_on) ? __ldg(lrow + hx) : -1;
        }
#pragma unroll
        for (int q = 0; q < RB; ++q) {
            const int r = r0 + q, y = ty0 - before + r;
            if (r >= SH) break;
            const int l4[4] = {v4[q].x, v4[q].y, v4[q].z, v4[q].w};
            uint32_t word = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t v = ((unsigned)l4[j] < (unsigned)a.n_labels) ? __ldg(a.decision + l4[j]) : 0u;
                word |= v << (8 * j);
            }
            *reinterpret_cast<uint32_t*>(s0 + r * DIL_PITCH + before + pad + 4 * lane) = word;
            if (PRE && r >= before && r < before + DIL_TH && y < a.ch) {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (l4[j] >= 0) a.pre[(size_t)y * a.cw + x4 + j] = ((word >> (8 * j)) & 1u) ? 255 : 0;
            }
            if (lane < k - 1) s0[r * DIL_PITCH + hs] = ((unsigned)vh[q] < (unsigned)a.n_labels) ? __ldg(a.decision + vh[q]) : 0;
        }
    }
    __syncthreads();
    // stage 2: output word j of row r = OR over d < k of the source bytes starting at s0 column pad + 4j + d
    for (int i = threadIdx.x; i < SH * (DIL_TW / 4); i += 256) {
        const int r = i / (DIL_TW / 4), j = i - r * (DIL_TW / 4);
        const uint32_t* row = reinterpret_cast<const uint32_t*>(s0 + r * DIL_PITCH) + j;
        uint32_t acc = 0;
        if (KF > 0) {
            constexpr int NW = (3 + (KF > 0 ? KF : 1) - 1) / 4 + 2;      // words that can be touched
            uint32_t w[NW];
#pragma unroll
            for (int q = 0; q < NW; ++q) w[q] = row[q];
#pragma unroll
            for (int d = 0; d < (KF > 0 ? KF : 1); ++d) {
                // byte offset pad + d: pad is block-uniform, so the word pick is a uniform select
                const int o = pad + d;
                uint32_t lo = w[0], hi = w[1];
#pragma unroll
                for (int q = 1; q < NW - 1; ++q)
                    if ((o >> 2) == q) { lo = w[q]; hi = w[q + 1]; }
                acc |= __funnelshift_r(lo, hi, 8 * (o & 3));
            }
        } else {
            int wi = pad >> 2, sh = (pad & 3) * 8;      // pad < 4: wi = 0
            uint32_t lo = row[wi], hi = row[wi + 1];
            for (int d = 0; d < k; ++d) {
                acc |= __funnelshift_r(lo, hi, sh);
                sh += 8;
                if (sh == 32) { sh = 0; ++wi; lo = hi; hi = row[wi + 1]; }
            }
        }
        reinterpret_cast<uint32_t*>(s1)[i] = acc;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < DIL_TH * DIL_TW / 4; i += 256) {
        const int r = i / (DIL_TW / 4), c = (i - r * (DIL_TW / 4)) * 4;
        const int y = ty0 + r, x = tx0 + c;
        if (y >= a.ch || x >= a.cw) continue;
        uint32_t v = 0;
        if (KF > 0) {
#pragma unroll
            for (int d = 0; d < (KF > 0 ? KF : 1); ++d) v |= *reinterpret_cast<const uint32_t*>(s1 + (r + d) * DIL_TW + c);
        } else {
            for (int d = 0; d < k; ++d) v |= *reinterpret_cast<const uint32_t*>(s1 + (r + d) * DIL_TW + c);
        }
        // bytes are 0/1 -> 0/255
        v = (v & 0x01010101u) * 255u;
        uint8_t* dst = a.mask + (size_t)(a.cy + y) * a.mask_stride + (a.cx + x);
        if (x + 3 < a.cw && (reinterpret_cast<uintptr_t>(dst) & 3) == 0) *reinterpret_cast<uint32_t*>(dst) = v;
        else
            for (int j = 0; j < 4 && x + j < a.cw; ++j) dst[j] = (uint8_t)(v >> (8 * j));
    }
}

// K5 -----------------------------------------------------------------------------
// counts[0] += #(m != 0 && t != 0), counts[1] += #(m != 0 || t != 0) (benchmark.py:12-13);
// truth either gray or BGR (converted like cv.cvtColor(BGR2GRAY), main.py:285).
// Gray truth with 16-byte aligned rows is read 16 pixels per thread.
// valid = {x, y, w, h}: the mask plane only counts inside this rectangle, everything outside reads as 0 (a sequence
// that moves its crop from frame to frame does not have to clear the plane in between); valid.z < 0: whole plane.
__global__ void __launch_bounds__(256) iou_kernel(const uint8_t* __restrict__ mask, long long mask_stride,
                                                  const uint8_t* __restrict__ truth, long long truth_stride,
                                                  int truth_channels, int h, int w, int4 valid,
                                                  unsigned long long* __restrict__ counts) {
    grid_launch_dependents();   // the next frame's K0 may start now: it touches nothing K3 or this kernel uses
    grid_dependency_wait();
    unsigned inter = 0, uni = 0;
    const bool vec = truth_channels == 1 && (w % 16 == 0) && (mask_stride % 16 == 0) && (truth_stride % 16 == 0) &&
                     ((reinterpret_cast<uintptr_t>(mask) | reinterpret_cast<uintptr_t>(truth)) & 15) == 0;
    if (vec) {
        const int per_row = w / 16;
        const long long n = (long long)h * per_row;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
            const int r = (int)(i / per_row), c = (int)(i - (long long)r * per_row) * 16;
            uint4 m = make_uint4(0u, 0u, 0u, 0u);
            const bool row_in = valid.z < 0 || (r >= valid.y && r < valid.y + valid.w);
            if (row_in && (valid.z < 0 || (c + 16 > valid.x && c < valid.x + valid.z))) {
                m = __ldg(reinterpret_cast<const uint4*>(mask + (size_t)r * mask_stride + c));
                if (valid.z >= 0 && (c < valid.x || c + 16 > valid.x + valid.z)) {       // chunk straddles the rectangle's edge
                    uint32_t* mw = reinterpret_cast<uint32_t*>(&m);
#pragma unroll
                    for (int b = 0; b < 16; ++b)
                        if (c + b < valid.x || c + b >= valid.x + valid.z) mw[b >> 2] &= ~(0xffu << (8 * (b & 3)));
                }
            }
            const uint4 t = __ldg(reinterpret_cast<const uint4*>(truth + (size_t)r * truth_stride + c));
            const uint32_t mm[4] = {m.x, m.y, m.z, m.w}, tt[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t a = __vcmpne4(mm[j], 0u), b = __vcmpne4(tt[j], 0u);   // 0xff per non-zero byte
                inter += __popc(a & b) >> 3;
                uni += __popc(a | b) >> 3;
            }
        }
    } else {
        const long long n = (long long)h * w;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
            const int r = (int)(i / w), c = (int)(i - (long long)r * w);
            const bool in = valid.z < 0 || (r >= valid.y && r < valid.y + valid.w && c >= valid.x && c < valid.x + valid.z);
            const bool m = in && mask[(size_t)r * mask_stride + c] != 0;
            const uint8_t* tp = truth + (size_t)r * truth_stride + (size_t)c * truth_channels;
            const bool t = (truth_channels == 3) ? (bgr2gray_px(tp[0], tp[1], tp[2]) != 0) : (tp[0] != 0);
            inter += m && t;
            uni += m || t;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        inter += __shfl_xor_sync(0xffffffffu, inter, o);
        uni += __shfl_xor_sync(0xffffffffu, uni, o);
    }
    __shared__ unsigned s_i[8], s_u[8];
    const int lane = threadIdx.x & 31;
    if (lane == 0) { s_i[threadIdx.x >> 5] = inter; s_u[threadIdx.x >> 5] = uni; }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long ti = 0, tu = 0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { ti += s_i[i]; tu += s_u[i]; }
        if (ti) atomicAdd(counts, ti);
        if (tu) atomicAdd(counts + 1, tu);
    }
}

// parity taps ----------------------------------------------------------------------
__global__ void __launch_bounds__(256) convert_kernel(const uint8_t* __restrict__ bgr, long long stride, int h, int w,
                                                      int space, const ColorTables* __restrict__ tab,
                                                      uint8_t* __restrict__ out, long long out_stride) {
    const long long n = (long long)h * w;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(i / w), c = (int)(i - (long long)r * w);
        const uint8_t* px = bgr + (size_t)r * stride + 3 * (size_t)c;
        int c0, c1, c2;
        if (space == 1) bgr2hsv_px(px[0], px[1], px[2], tab->sdiv, tab->hdiv, c0, c1, c2);
        else if (space == 2) bgr2lab_px(px[0], px[1], px[2], tab->gamma, tab->cbrt_tab, c0, c1, c2);
        else { c0 = px[0]; c1 = px[1]; c2 = px[2]; }
        uint8_t* o = out + (size_t)r * out_stride + 3 * (size_t)c;
        o[0] = (uint8_t)c0; o[1] = (uint8_t)c1; o[2] = (uint8_t)c2;
    }
}

// X[row, q*3K + 3k + ch] = plane value at (r + dr_k, c + dc_k) or -1 outside the crop (:263-272)
__global__ void __launch_bounds__(256) gather_kernel(const uint8_t* __restrict__ frame, long long stride, int cx, int cy,
                                                     int cw, int ch, Geom g, const ColorTables* __restrict__ tab,
                                                     int16_t* __restrict__ X) {
    const long long n = (long long)ch * cw * g.K;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(i % g.K);
        const long long pix = i / g.K;
        const int r = (int)(pix / cw), c = (int)(pix - (long long)r * cw);
        int dr, dc;
        star_tap(k, dr, dc);
        const int rr = r + dr, cc = c + dc;
        const bool ok = rr >= 0 && rr < ch && cc >= 0 && cc < cw;
        int b = 0, gg = 0, red = 0;
        if (ok) {
            const uint8_t* px = frame + (size_t)(cy + rr) * stride + 3 * (size_t)(cx + cc);
            b = px[0]; gg = px[1]; red = px[2];
        }
        for (int q = 0; q < g.n_spaces; ++q) {
            int c0 = -1, c1 = -1, c2 = -1;
            if (ok) {
                const int sid = g.space_id[q];
                if (sid == 1) bgr2hsv_px(b, gg, red, tab->sdiv, tab->hdiv, c0, c1, c2);
                else if (sid == 2) bgr2lab_px(b, gg, red, tab->gamma, tab->cbrt_tab, c0, c1, c2);
                else { c0 = b; c1 = gg; c2 = red; }
            }
            int16_t* o = X + (size_t)pix * g.F + (size_t)q * 3 * g.K + 3 * k;
            o[0] = (int16_t)c0; o[1] = (int16_t)c1; o[2] = (int16_t)c2;
        }
    }
}

}  // namespace pcm
