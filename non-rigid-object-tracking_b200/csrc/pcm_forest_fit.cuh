// pcm_forest_fit.cuh -- random-forest TRAINING on the GPU (sm_100a), tree for tree the forest that
//     RandomForestClassifier(random_state=42, n_estimators, max_depth).fit(X / 255, labels)
// of the reference's addModel grows (maskers/pixel_classification.py:199-200), as scikit-learn 1.9.0 builds it
// (sklearn/tree/_tree.pyx DepthFirstTreeBuilder, _splitter.pyx node_split_best, _criterion.pyx Gini;
// file:line in oracle/forest_fit_oracle.c, whose restatement is pinned against scikit-learn itself).
//
// What makes an exact GPU version possible: the features of this path are integers v in {-1..255} (X / 255 cast to
// float32 takes 257 distinct values), the two classes and the bootstrap counts are integers.  scikit-learn sorts
// a node's samples by one feature and scans the sorted run; here the node's samples are binned into a 257-bin
// histogram of weighted class counts (shared-memory atomics) and the bins are scanned in ascending order -- the
// same candidate positions, the same integer sums at each of them and therefore the same float64 impurity
// expressions (evaluated with explicit round-to-nearest operations, no FMA contraction).  The pseudo-random feature
// draw (Fisher-Yates on the `features` permutation with xorshift `our_rand_r`, constant-feature bookkeeping carried
// from node to node in depth-first order) is inherently sequential per tree and is reproduced step for step.
//
// One CTA grows one tree; a forest (and several forests on several streams) fill the GPU.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace pcm {

constexpr int FIT_THREADS = 256;
constexpr int FIT_BINS = 257;              // value v in -1..255 -> bin v + 1
constexpr int FIT_MAX_DEPTH = 24;
constexpr int FIT_MAX_FEATURES = 1176;     // 3 spaces x 3 channels x (1 + 8 * 16) taps, rounded up

// sample entry: row index (24 bits) | class (1 bit) | bootstrap count (7 bits)
__host__ __device__ inline uint32_t fit_pack(uint32_t idx, uint32_t y, uint32_t w) { return idx | (y << 24) | (w << 25); }

struct FitArgs {
    const int16_t* Xt;          // [F][n_pad] feature-major rows (v in -1..255)
    long long n_pad;
    const uint8_t* y;           // [n] 0/1
    const uint8_t* counts;      // [T][n] bootstrap counts of tree t
    const uint32_t* rand_state; // [T] splitter seeds
    int n, F, max_depth, max_features, cap;   // cap = node capacity per tree
    uint32_t* samples;          // [T][n] scratch
    uint32_t* tmp;              // [T][n] scratch
    // outputs, tree t at [t * cap, (t + 1) * cap)
    int32_t* feature;           // -2 leaf
    double* threshold;          // -2.0 leaf
    int32_t* left;              // -1 leaf
    int32_t* right;
    double* value1;             // class-1 fraction of the node's weighted samples
    int32_t* n_node_samples;
    int32_t* node_count;        // [T]; -1 = capacity exceeded
};

__device__ __forceinline__ uint32_t fit_rand_r(uint32_t& s) {
    if (s == 0) s = 1;
    s ^= s << 13;
    s ^= s >> 17;
    s ^= s << 5;
    return s % 2147483648u;
}

// Gini impurity of a node with class sums c0, c1 and weight w (= c0 + c1), in scikit-learn's evaluation order
__device__ __forceinline__ double fit_gini(double c0, double c1, double w) {
    const double sq = __dadd_rn(__dmul_rn(c0, c0), __dmul_rn(c1, c1));
    return __dsub_rn(1.0, __ddiv_rn(sq, __dmul_rn(w, w)));
}

struct FitStack {
    int start, end, depth, parent, is_left, n_constant, t0, t1;
    double impurity;
};

// [n][F] row-major -> [F][n_pad] feature-major (32 x 32 tiles through shared memory)
__global__ void __launch_bounds__(256) fit_transpose_kernel(const int16_t* __restrict__ X, int n, int F,
                                                            int16_t* __restrict__ Xt, long long n_pad) {
    __shared__ int16_t tile[32][33];
    const int r0 = blockIdx.x * 32, f0 = blockIdx.y * 32;
    for (int k = threadIdx.y; k < 32; k += 8) {
        const int r = r0 + k, f = f0 + threadIdx.x;
        tile[k][threadIdx.x] = (r < n && f < F) ? X[(size_t)r * F + f] : (int16_t)0;
    }
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += 8) {
        const int f = f0 + k, r = r0 + threadIdx.x;
        if (f < F && r < n) Xt[(size_t)f * n_pad + r] = tile[threadIdx.x][k];
    }
}

__global__ void __launch_bounds__(FIT_THREADS) forest_fit_kernel(const FitArgs a) {
    __shared__ int hist[2][FIT_BINS + 31];
    __shared__ int16_t features[FIT_MAX_FEATURES], constant_features[FIT_MAX_FEATURES];
    __shared__ FitStack stack[FIT_MAX_DEPTH + 4];
    __shared__ int s_cur_feature, s_cl, s_cr, s_sp, s_red[2][FIT_THREADS / 32];
    // state of the split search of the current node (written by thread 0 only)
    __shared__ int s_best_feature, s_best_bin, s_best_next, s_best_l0, s_best_l1;
    __shared__ double s_best_proxy;
    __shared__ int s_fi, s_fj, s_visited, s_found, s_drawn, s_total_constants;
    __shared__ uint32_t s_rand;

    const int t = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = a.n, F = a.F;
    uint32_t* samples = a.samples + (size_t)t * n;
    uint32_t* tmp = a.tmp + (size_t)t * n;
    const uint8_t* counts = a.counts + (size_t)t * n;
    const size_t ob = (size_t)t * a.cap;

    for (int f = tid; f < F; f += FIT_THREADS) features[f] = (int16_t)f;
    if (tid == 0) { s_cl = 0; s_rand = a.rand_state[t]; }
    __syncthreads();
    // samples with a non-zero bootstrap count (Splitter.init); their order is irrelevant: every quantity below
    // is a sum of integers over a SET of samples
    int c0 = 0, c1 = 0;
    for (int base = 0; base < n; base += FIT_THREADS) {
        const int i = base + tid;
        const uint32_t w = i < n ? counts[i] : 0u;
        const uint32_t yy = i < n ? a.y[i] : 0u;
        const unsigned m = __ballot_sync(0xffffffffu, w != 0);
        int pos = 0;
        if (lane == 0 && m) pos = atomicAdd(&s_cl, __popc(m));
        pos = __shfl_sync(0xffffffffu, pos, 0);
        if (w) {
            samples[pos + __popc(m & ((1u << lane) - 1))] = fit_pack((uint32_t)i, yy, w);
            if (yy) c1 += (int)w; else c0 += (int)w;
        }
    }
    c0 = __reduce_add_sync(0xffffffffu, c0);
    c1 = __reduce_add_sync(0xffffffffu, c1);
    if (lane == 0) { s_red[0][warp] = c0; s_red[1][warp] = c1; }
    __syncthreads();
    int node_count = 0;
    double weighted_n_samples = 0.0;
    {
        int T0 = 0, T1 = 0;
        for (int w = 0; w < FIT_THREADS / 32; ++w) { T0 += s_red[0][w]; T1 += s_red[1][w]; }
        weighted_n_samples = (double)(T0 + T1);
        if (tid == 0) {
            stack[0] = FitStack{0, s_cl, 0, -1, 0, 0, T0, T1, fit_gini((double)T0, (double)T1, (double)(T0 + T1))};
            s_sp = 1;
        }
    }
    __syncthreads();

    while (s_sp > 0) {
        const FitStack r = stack[s_sp - 1];
        __syncthreads();                                  // everybody has read the record before it is replaced
        const int start = r.start, end = r.end, nn = end - start;
        const double t0 = (double)r.t0, t1 = (double)r.t1, W = (double)(r.t0 + r.t1);
        const double EPS = 2.220446049250313e-16;
        bool is_leaf = r.depth >= a.max_depth || nn < 2 || r.impurity <= EPS;
        if (tid == 0) {
            s_sp--;
            s_best_feature = -1; s_best_proxy = -INFINITY;
            s_fi = F; s_visited = 0; s_found = 0; s_drawn = 0; s_total_constants = r.n_constant;
        }
        if (!is_leaf) {
            const int n_known = r.n_constant;
            for (;;) {
                // ---- draw (thread 0): Fisher-Yates step(s) until a feature has to be evaluated or the loop ends ----
                if (tid == 0) {
                    int cur = -1;
                    while (s_fi > s_total_constants &&
                           (s_visited < a.max_features || s_visited <= s_found + s_drawn)) {
                        s_visited++;
                        uint32_t rs = s_rand;
                        int fj = s_drawn + (int)(fit_rand_r(rs) % (uint32_t)(s_fi - s_found - s_drawn));
                        s_rand = rs;
                        if (fj < n_known) {
                            const int16_t x = features[s_drawn]; features[s_drawn] = features[fj]; features[fj] = x;
                            s_drawn++;
                            continue;
                        }
                        fj += s_found;
                        s_fj = fj;
                        cur = features[fj];
                        break;
                    }
                    s_cur_feature = cur;
                }
                for (int b = tid; b < 2 * (FIT_BINS + 31); b += FIT_THREADS) (&hist[0][0])[b] = 0;
                __syncthreads();
                const int cf = s_cur_feature;
                if (cf < 0) break;
                // ---- weighted class histogram of the node's samples over the feature's 257 values ----
                const int16_t* col = a.Xt + (size_t)cf * a.n_pad;
                for (int p = start + tid; p < end; p += FIT_THREADS) {
                    const uint32_t e = samples[p];
                    const int b = (int)col[e & 0xffffffu] + 1;
                    atomicAdd(&hist[(e >> 24) & 1u][b], (int)(e >> 25));
                }
                __syncthreads();
                // ---- scan (warp 0): 9 bins per lane, candidates in ascending value order ----
                if (warp == 0) {
                    int h0[9], h1[9];
                    int s0 = 0, s1 = 0, nz = 0;
#pragma unroll
                    for (int k = 0; k < 9; ++k) {
                        h0[k] = hist[0][9 * lane + k]; h1[k] = hist[1][9 * lane + k];
                        s0 += h0[k]; s1 += h1[k];
                        nz += (h0[k] + h1[k]) != 0;
                    }
                    int p0 = s0, p1 = s1;                 // inclusive prefix over lanes
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int u0 = __shfl_up_sync(0xffffffffu, p0, o), u1 = __shfl_up_sync(0xffffffffu, p1, o);
                        if (lane >= o) { p0 += u0; p1 += u1; }
                    }
                    const int nonempty = __reduce_add_sync(0xffffffffu, nz);
                    int l0 = p0 - s0, l1 = p1 - s1;       // class sums strictly below this lane's bins
                    double best = -INFINITY;
                    int best_bin = 0x7fffffff, bl0 = 0, bl1 = 0;
                    if (nonempty > 1) {
#pragma unroll
                        for (int k = 0; k < 9; ++k) {
                            if (h0[k] + h1[k] == 0) continue;
                            l0 += h0[k]; l1 += h1[k];
                            if (l0 + l1 >= r.t0 + r.t1) continue;      // nothing to the right: not a split position
                            const double dl0 = (double)l0, dl1 = (double)l1, wl = (double)(l0 + l1);
                            const double wr = __dsub_rn(W, wl);
                            const double gl = fit_gini(dl0, dl1, wl);
                            const double gr = fit_gini(__dsub_rn(t0, dl0), __dsub_rn(t1, dl1), wr);
                            const double proxy = __dsub_rn(__dmul_rn(-wr, gr), __dmul_rn(wl, gl));
                            if (proxy > best) { best = proxy; best_bin = 9 * lane + k; bl0 = l0; bl1 = l1; }
                        }
                    }
                    // warp arg-max, ties to the smaller bin (= first encountered in scikit-learn's scan)
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        const double ob_ = __shfl_xor_sync(0xffffffffu, best, o);
                        const int obin = __shfl_xor_sync(0xffffffffu, best_bin, o);
                        const int o0 = __shfl_xor_sync(0xffffffffu, bl0, o), o1 = __shfl_xor_sync(0xffffffffu, bl1, o);
                        if (ob_ > best || (ob_ == best && obin < best_bin)) { best = ob_; best_bin = obin; bl0 = o0; bl1 = o1; }
                    }
                    // first non-empty bin above best_bin (the upper neighbour of the threshold)
                    int nxt = 0x7fffffff;
#pragma unroll
                    for (int k = 8; k >= 0; --k)
                        if (h0[k] + h1[k] != 0 && 9 * lane + k > best_bin) nxt = 9 * lane + k;
                    nxt = __reduce_min_sync(0xffffffffu, nxt);
                    if (lane == 0) {
                        const int fj = s_fj;
                        if (nonempty <= 1) {              // constant in this node (max - min <= FEATURE_THRESHOLD)
                            const int16_t x = features[fj]; features[fj] = features[s_total_constants]; features[s_total_constants] = x;
                            s_found++; s_total_constants++;
                        } else {
                            s_fi--;
                            const int16_t x = features[s_fi]; features[s_fi] = features[fj]; features[fj] = x;
                            if (best > s_best_proxy) {
                                s_best_proxy = best; s_best_feature = cf; s_best_bin = best_bin; s_best_next = nxt;
                                s_best_l0 = bl0; s_best_l1 = bl1;
                            }
                        }
                    }
                }
                __syncthreads();
            }
            // restore the known constants' order, publish the newly found ones (node_split_best :491-499)
            for (int f = tid; f < n_known; f += FIT_THREADS) features[f] = constant_features[f];
            __syncthreads();
            for (int f = n_known + tid; f < n_known + s_found; f += FIT_THREADS) constant_features[f] = features[f];
            __syncthreads();
        }
        // ---- partition + node record ----
        int pos = end;
        const bool found = !is_leaf && s_best_feature >= 0;
        double imp_l = 0.0, imp_r = 0.0, improvement = 0.0;
        if (found) {
            const int bf = s_best_feature, bb = s_best_bin;
            const int16_t* col = a.Xt + (size_t)bf * a.n_pad;
            if (tid == 0) { s_cl = 0; s_cr = 0; }
            __syncthreads();
            for (int base = start; base < end; base += FIT_THREADS) {
                const int p = base + tid;
                const bool ok = p < end;
                const uint32_t e = ok ? samples[p] : 0u;
                const bool go_left = ok && ((int)col[e & 0xffffffu] + 1 <= bb);
                const unsigned ml = __ballot_sync(0xffffffffu, go_left), mr = __ballot_sync(0xffffffffu, ok && !go_left);
                int pl = 0, pr = 0;
                if (lane == 0) {
                    if (ml) pl = atomicAdd(&s_cl, __popc(ml));
                    if (mr) pr = atomicAdd(&s_cr, __popc(mr));
                }
                pl = __shfl_sync(0xffffffffu, pl, 0);
                pr = __shfl_sync(0xffffffffu, pr, 0);
                const unsigned below = (1u << lane) - 1;
                if (go_left) tmp[start + pl + __popc(ml & below)] = e;
                else if (ok) tmp[end - 1 - (pr + __popc(mr & below))] = e;
            }
            __syncthreads();
            for (int p = start + tid; p < end; p += FIT_THREADS) samples[p] = tmp[p];
            pos = start + s_cl;
            const double l0 = (double)s_best_l0, l1 = (double)s_best_l1, wl = (double)(s_best_l0 + s_best_l1);
            const double wr = __dsub_rn(W, wl);
            imp_l = fit_gini(l0, l1, wl);
            imp_r = fit_gini(__dsub_rn(t0, l0), __dsub_rn(t1, l1), wr);
            improvement = __dmul_rn(__ddiv_rn(W, weighted_n_samples),
                                    __dsub_rn(__dsub_rn(r.impurity, __dmul_rn(__ddiv_rn(wr, W), imp_r)),
                                              __dmul_rn(__ddiv_rn(wl, W), imp_l)));
        }
        if (!is_leaf) is_leaf = pos >= end || __dadd_rn(improvement, EPS) < 0.0;
        const int id = node_count++;
        if (id >= a.cap) { if (tid == 0) a.node_count[t] = -1; return; }
        if (tid == 0) {
            if (r.parent >= 0) { if (r.is_left) a.left[ob + r.parent] = id; else a.right[ob + r.parent] = id; }
            a.left[ob + id] = -1; a.right[ob + id] = -1;
            a.feature[ob + id] = is_leaf ? -2 : s_best_feature;
            double thr = -2.0;
            if (!is_leaf) {
                const float lo = (float)((double)(s_best_bin - 1) / 255.0), hi = (float)((double)(s_best_next - 1) / 255.0);
                thr = __dadd_rn(__ddiv_rn((double)lo, 2.0), __ddiv_rn((double)hi, 2.0));
            }
            a.threshold[ob + id] = thr;
            a.value1[ob + id] = __ddiv_rn(t1, W);
            a.n_node_samples[ob + id] = nn;
            if (!is_leaf) {
                const int tc = s_total_constants;
                stack[s_sp++] = FitStack{pos, end, r.depth + 1, id, 0, tc, r.t0 - s_best_l0, r.t1 - s_best_l1, imp_r};
                stack[s_sp++] = FitStack{start, pos, r.depth + 1, id, 1, tc, s_best_l0, s_best_l1, imp_l};
            }
        }
        __syncthreads();
    }
    if (tid == 0) a.node_count[t] = node_count;
}

// ---- PCA novelty detector of addModel (:203-213) on the resident training rows -------------------------------
// Gram matrix and column sums of the class-1 rows: G[i][j] = sum_r y_r v_ri v_rj, S[i] = sum_r y_r v_ri (raw integer
// feature values v; exact: products < 2^16, every partial sum an integer far below 2^53).  The host turns them into
// sklearn's covariance (decomposition/_pca.py `_fit_full`, solver covariance_eigh: C = X^T X - n mean mean^T,
// C /= n - 1) and takes the leading eigenvector.  One block = a 32 x 32 tile of G, rows in chunks of 64.
__global__ void __launch_bounds__(256) pca_gram_kernel(const int16_t* __restrict__ Xt, long long n_pad, const uint8_t* __restrict__ y,
                                                       int n, int F, double* __restrict__ G, double* __restrict__ S,
                                                       unsigned long long* __restrict__ n1) {
    __shared__ int A[32][65], B[32][65];
    const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;          // 16 x 16 threads, 2 x 2 outputs each
    long long acc[2][2] = {{0, 0}, {0, 0}};
    long long colsum = 0, ones = 0;
    for (int r0 = 0; r0 < n; r0 += 64) {
        for (int k = threadIdx.x; k < 32 * 64; k += 256) {
            const int f = k >> 6, r = r0 + (k & 63);
            const int m = (r < n) ? (int)y[r] : 0;
            A[f][k & 63] = (m && i0 + f < F) ? (int)Xt[(size_t)(i0 + f) * n_pad + r] : 0;
            B[f][k & 63] = (m && j0 + f < F) ? (int)Xt[(size_t)(j0 + f) * n_pad + r] : 0;
        }
        __syncthreads();
        int c[2][2] = {{0, 0}, {0, 0}};
#pragma unroll 16
        for (int k = 0; k < 64; ++k) {
            const int a0 = A[2 * ty][k], a1 = A[2 * ty + 1][k], b0 = B[2 * tx][k], b1 = B[2 * tx + 1][k];
            c[0][0] += a0 * b0; c[0][1] += a0 * b1; c[1][0] += a1 * b0; c[1][1] += a1 * b1;
        }
        acc[0][0] += c[0][0]; acc[0][1] += c[0][1]; acc[1][0] += c[1][0]; acc[1][1] += c[1][1];
        if (blockIdx.x == 0 && threadIdx.x < 32) {                    // column sums of the i-tile, class-1 count
            int sm = 0;
            for (int k = 0; k < 64; ++k) sm += A[threadIdx.x][k];
            colsum += sm;
            if (blockIdx.y == 0 && threadIdx.x == 0)
                for (int k = 0; k < 64 && r0 + k < n; ++k) ones += y[r0 + k];
        }
        __syncthreads();
    }
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            const int i = i0 + 2 * ty + u, j = j0 + 2 * tx + v;
            if (i < F && j < F) G[(size_t)i * F + j] = (double)acc[u][v];
        }
    if (blockIdx.x == 0 && threadIdx.x < 32 && i0 + (int)threadIdx.x < F) S[i0 + threadIdx.x] = (double)colsum;
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *n1 = (unsigned long long)ones;
}

// L1 reconstruction error of EVERY training row under a PCA of KC components (:208-211), x = v / 255:
//   t_j = x . c_j - mean . c_j  (both dot products fma-accumulated in feature order)
//   err = sum_f |x_f - r_f|,  r_f = fma(t_{KC-1}, c_{KC-1,f}, ... fma(t_0, c_0f, mean_f))
// For KC = 1 this is the rank-1 arithmetic t = x . c - mean . c, err = sum_f |x_f - fma(t, c_f, mean_f)|.  One thread per row.
template <int KC>
__global__ void __launch_bounds__(256) pca_residual_kernel(const int16_t* __restrict__ Xt, long long n_pad, int n, int F,
                                                           const double* __restrict__ mean, const double* __restrict__ comp,
                                                           double* __restrict__ err) {
    extern __shared__ double sh[];          // comp[KC][F] | mean[F]
    for (int f = threadIdx.x; f < (KC + 1) * F; f += blockDim.x) sh[f] = f < KC * F ? comp[f] : mean[f - KC * F];
    __syncthreads();
    const double* shm = sh + KC * F;
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double t[KC], mdc[KC];
#pragma unroll
    for (int j = 0; j < KC; ++j) { t[j] = 0.0; mdc[j] = 0.0; }
    for (int f = 0; f < F; ++f) {
        const double x = (double)Xt[(size_t)f * n_pad + r] / 255.0;
#pragma unroll
        for (int j = 0; j < KC; ++j) {
            t[j] = fma(x, sh[j * F + f], t[j]);
            mdc[j] = fma(shm[f], sh[j * F + f], mdc[j]);
        }
    }
#pragma unroll
    for (int j = 0; j < KC; ++j) t[j] -= mdc[j];
    double e = 0.0;
    for (int f = 0; f < F; ++f) {
        const double x = (double)Xt[(size_t)f * n_pad + r] / 255.0;
        double rec = shm[f];
#pragma unroll
        for (int j = 0; j < KC; ++j) rec = fma(t[j], sh[j * F + f], rec);
        e += fabs(x - rec);
    }
    err[r] = e;
}

}  // namespace pcm
