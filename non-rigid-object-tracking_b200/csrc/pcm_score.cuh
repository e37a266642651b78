// pcm_score.cuh -- K0 (colour planes) and K1 (fused star features + forests) of the PC masker hot path (sm_100a).
// Templates only: included by pcm_kernels.cuh (all kernels, one translation unit: pcm_api.cu) and by
// pcm_score_inst.cu, which instantiates score_kernel once per tile height in its own translation unit so
// that the instantiations compile in parallel.
//
//  K0 planes_kernel       BGR crop -> planar HSV/LAB/BGR planes + validity plane (cvtColor :294-309)
//  K1 score_kernel        TMA tiles of those planes (smem, halo) -> star taps -> forest(s)
//                         [-> PCA novelty error] [-> temporal blend] -> P(fg) f64 [, err f64]
//                         (a PCA of two or more components: the error map of novelty_kernel, pcm_kernels.cuh)
//                         replaces cvtColor + getFeatures + X/255 + predict_proba + PCA
//                         (reference maskers/pixel_classification.py:53-63, :80-95)
//                         epilogue: per-label sums / areas (np.unique :97 + first loop of
//                         compileSaliencyMap :235-238), warp-aggregated atomics
//  K2 segment_decide      per-label score and decision (:240-242); labels inside the guard
//                         band are re-evaluated exactly (sequential float32, raster order)
//  K3 mask_dilate         decision -> 0/255 map (:242-246) fused with cv.dilate (:112)
//  K5 iou_kernel          computeBenchmark counts (benchmark.py:8-14)
//  + convert_kernel / gather_kernel: parity taps (pcm_convert, pcm_gather_features)
#pragma once
#include "pcm_device.cuh"
#include <cuda.h>

namespace pcm {

// ------------------------------------------------------------------------------
// packed forest (built on the host by Encoder in pcm_api.cu)
//   Every tree owns a contiguous run of fixed-size entries (NodeT): internal nodes and one
//   self-looping pseudo-node per leaf, laid out breadth-first so that the two children of a
//   node are ADJACENT entries (left, then right).  The traversal is branch-free and a thread
//   that has reached a leaf simply stays there.
//     tap   byte offset of the tested value inside the plane tile
//     thr   the value v (u8, 0 outside the crop) goes RIGHT iff v > thr
//     left  byte offset of the LEFT child's entry from the start of the forest's entry
//           array (right child = + NODE_BYTES); relocated to an absolute shared-memory
//           address when the forest is staged in shared memory
//     leaf pseudo-node: tap = 0, thr = LEAF_THR (never right), left = self
//   leaves[i] = class-1 fraction of entry i (leaf entries; 0 elsewhere), parallel array
//   trees[t] = {root entry offset (bytes), depth, -, -}   (only the offset is used, and only
//              for trees beyond MAX_TOP_TREES)
// The crop-border sentinel -1 of the reference (:263) is handled by the encoder:
// nodes with integer threshold -1 test the validity plane instead (0 outside the crop).
// ------------------------------------------------------------------------------
// 8-byte entries; a 16-byte {tap, thr, left, -} layout (LDS.128, one ALU op fewer per visit) was
// measured 22 % slower: the shared-memory pipe saturates (profiles/README.md).
typedef uint2 NodeT;   // {tap << 16 | thr, left}
__host__ __device__ inline NodeT make_node(unsigned tap, unsigned thr, unsigned left) { return make_uint2((tap << 16) | thr, left); }
__host__ __device__ inline unsigned node_tap(const NodeT& n) { return n.x >> 16; }
__host__ __device__ inline unsigned node_thr(const NodeT& n) { return n.x & 0xffffu; }
__host__ __device__ inline unsigned node_left(const NodeT& n) { return n.y; }
__host__ __device__ inline void node_set_left(NodeT& n, unsigned v) { n.y = v; }
constexpr unsigned LEAF_THR = 0xffffu;
constexpr unsigned NODE_BYTES = sizeof(NodeT);

struct DevForest {
    const NodeT* nodes;      // [n_nodes] entries
    const double* leaves;    // [n_nodes] values, parallel to nodes
    const int4* trees;
    int n_trees, n_nodes, n_leaves;
};

// Root and its two children of the first MAX_TOP_TREES trees, passed in the kernel
// parameter (constant) bank: the first two levels of a tree are evaluated from
// warp-uniform operands, without touching the shared-memory pipe for node fetches
// (entry.y here is still forest-relative).
constexpr int MAX_TOP_TREES = 48;
struct TopNodes {
    NodeT n[MAX_TOP_TREES][3];   // {root, left child, right child}
};

struct DevPCA {
    const double* comp;      // components_[0][F]
    const double* comp255;   // components_[0][F] / 255
    const double* mean;      // mean_[F]
    double mean_dot_comp;    // mean_ . components_[0]
};

// ---- K0: BGR crop -> planar colour planes + validity plane ------------------------------
// planes[p][r][c], p = 3*q + channel in `features` token order, last plane = 1 (inside the
// crop).  Rows are `pitch` bytes apart (multiple of 16 so that TMA can tile the tensor);
// the tile loads of K1 zero-fill everything outside [0,cw) x [0,ch).
struct PlanesArgs {
    const uint8_t* frame;
    long long stride;
    int cx, cy, cw, ch;
    Geom g;
    const ColorTables* tables;
    uint8_t* planes;
    long long pitch;          // bytes between rows
    long long plane_stride;   // BYTES between planes
    unsigned* tile_counter;   // reset here for K1's dynamic tile scheduler
    // per-label accumulators of K2, reset here (saves three memset launches per frame)
    int n_labels;
    double* sum;
    double* asum;
    int* area;
    int* rmin;
    int* rmax;
    int* cmin;
    int* cmax;
    int* n_flagged;
    int early;                // 1: the predecessor on the stream is this handle's own K3 / K5 (see below)
    int reset_flagged;        // 1: first K0 launch of a frame (a frame fed in row bands has several; n_labels = 0 in the others)
};

// MODE 1: features "<n> hsv_lab" (config.yaml:30), MODE 2: "<n> lab" (benchmark.py:48), MODE 0: any
// combination (space ids read per pixel).  FULL groups (four pixels inside the crop, 4-byte aligned
// source) take a path without per-pixel bounds checks.
template <int MODE>
__global__ void __launch_bounds__(256) planes_kernel(const PlanesArgs a) {
    __shared__ ColorTables tab;
    for (int i = threadIdx.x; i < (int)(sizeof(ColorTables) / 4); i += blockDim.x)
        reinterpret_cast<uint32_t*>(&tab)[i] = reinterpret_cast<const uint32_t*>(a.tables)[i];
    // Programmatic dependent launch.  a.early == 1 (the library enqueued this launch on the handle's
    // PRIVATE stream right behind its own mask_dilate / iou kernel): K0 does not wait for its
    // predecessor before it works.  It can only have been started by a K3 / K5 that is already running,
    // i.e. after the previous frame's K2 has completed (K3 releases its dependents after its own wait,
    // K5 at its very start), nothing K0 writes (planes, per-label accumulators, tile counter) is touched
    // by K3 or K5, and nobody else can have queued a producer of `frame` on that stream.  It waits at
    // its END instead, so that "K0 complete" still implies "everything before K0 complete" for K1.
    // a.early == 0 (caller-provided stream, or anything else queued last): the predecessor may be a
    // foreign kernel that writes `frame`, so K0 waits before it reads or resets anything.
    if (!a.early) grid_dependency_wait();
    grid_launch_dependents();
    if (blockIdx.x == 0 && threadIdx.x == 0) { *a.tile_counter = 0; if (a.reset_flagged) *a.n_flagged = 0; }
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.n_labels; i += gridDim.x * blockDim.x) {
        a.sum[i] = 0.0; a.asum[i] = 0.0; a.area[i] = 0; a.rmin[i] = 0x7fffffff; a.rmax[i] = -1;
        a.cmin[i] = 0x7fffffff; a.cmax[i] = -1;
    }
    __syncthreads();
    const int groups_per_row = (a.cw + 3) >> 2;
    const int n_groups = a.ch * groups_per_row;          // crop <= 2^30 px (validate_update)
    const int n_spaces = MODE == 1 ? 2 : (MODE == 2 ? 1 : a.g.n_spaces);
    const int nch = 3 * n_spaces;
    constexpr int NOUT = MODE == 1 ? 6 : (MODE == 2 ? 3 : 3 * MAX_SPACES);

    auto convert = [&](int b, int gg, int rr, int j, uint32_t (&out)[NOUT]) {
        if (MODE == 1 || MODE == 2) {
            int v0, v1, v2;
            if (MODE == 1) {
                bgr2hsv_px(b, gg, rr, tab.sdiv, tab.hdiv, v0, v1, v2);
                out[0] |= (uint32_t)v0 << (8 * j); out[1] |= (uint32_t)v1 << (8 * j); out[2] |= (uint32_t)v2 << (8 * j);
            }
            bgr2lab_px(b, gg, rr, tab.gamma, tab.cbrt_tab, v0, v1, v2);
            constexpr int o = MODE == 1 ? 3 : 0;
            out[o] |= (uint32_t)v0 << (8 * j); out[o + 1] |= (uint32_t)v1 << (8 * j); out[o + 2] |= (uint32_t)v2 << (8 * j);
        } else {
#pragma unroll
            for (int q = 0; q < MAX_SPACES; ++q) {
                if (q < n_spaces) {
                    int v0, v1, v2;
                    const int sid = a.g.space_id[q];
                    if (sid == 1) bgr2hsv_px(b, gg, rr, tab.sdiv, tab.hdiv, v0, v1, v2);
                    else if (sid == 2) bgr2lab_px(b, gg, rr, tab.gamma, tab.cbrt_tab, v0, v1, v2);
                    else { v0 = b; v1 = gg; v2 = rr; }
                    out[3 * q + 0] |= (uint32_t)v0 << (8 * j);
                    out[3 * q + 1] |= (uint32_t)v1 << (8 * j);
                    out[3 * q + 2] |= (uint32_t)v2 << (8 * j);
                }
            }
        }
    };

    // 4 pixels = 12 bytes: three aligned words when possible, byte loads otherwise.  The words of
    // the thread's NEXT group are requested before the current group is converted.
    auto fetch = [&](int r, int g, uint32_t (&w3)[3]) {      // group g of crop row r
        const int c0 = g * 4;
        const uint8_t* src = a.frame + (long long)(a.cy + r) * a.stride + (long long)(a.cx + c0) * 3;
        w3[0] = w3[1] = w3[2] = 0u;
        if (c0 + 3 < a.cw && (reinterpret_cast<uintptr_t>(src) & 3) == 0) {
#pragma unroll
            for (int q = 0; q < 3; ++q) w3[q] = __ldg(reinterpret_cast<const uint32_t*>(src) + q);
        } else {
#pragma unroll
            for (int q = 0; q < 12; ++q)
                if (c0 + q / 3 < a.cw) w3[q / 4] |= (uint32_t)__ldg(src + q) << (8 * (q % 4));
        }
    };
    // (row, group) of the thread's current and next group advance by a constant (dr, dg) per
    // iteration: no integer division in the loop
    const int stride = gridDim.x * blockDim.x;
    const int dr = stride / groups_per_row, dg = stride - dr * groups_per_row;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int r = i / groups_per_row, g = i - r * groups_per_row;
    int rn = r + dr, gn = g + dg;
    if (gn >= groups_per_row) { gn -= groups_per_row; ++rn; }
    uint32_t w3[3], nx[3] = {0u, 0u, 0u};
    if (i < n_groups) fetch(r, g, w3);
    for (; i < n_groups; i += stride) {
        if (i + stride < n_groups) fetch(rn, gn, nx);
        const int c0 = g * 4;
        uint32_t out[NOUT];
#pragma unroll
        for (int p = 0; p < NOUT; ++p) out[p] = 0;
        uint32_t valid = 0;
        const bool full = c0 + 3 < a.cw;
        if (full) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                convert((w3[(3 * j) / 4] >> (8 * ((3 * j) % 4))) & 0xff, (w3[(3 * j + 1) / 4] >> (8 * ((3 * j + 1) % 4))) & 0xff,
                        (w3[(3 * j + 2) / 4] >> (8 * ((3 * j + 2) % 4))) & 0xff, j, out);
            valid = 0x01010101u;
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (c0 + j < a.cw) {
                    convert((w3[(3 * j) / 4] >> (8 * ((3 * j) % 4))) & 0xff, (w3[(3 * j + 1) / 4] >> (8 * ((3 * j + 1) % 4))) & 0xff,
                            (w3[(3 * j + 2) / 4] >> (8 * ((3 * j + 2) % 4))) & 0xff, j, out);
                    valid |= 1u << (8 * j);
                }
            }
        }
        uint8_t* dst = a.planes + (long long)r * a.pitch + c0;
#pragma unroll
        for (int p = 0; p < NOUT; ++p)
            if (p < nch) *reinterpret_cast<uint32_t*>(dst + p * a.plane_stride) = out[p];
        *reinterpret_cast<uint32_t*>(dst + nch * a.plane_stride) = valid;
        w3[0] = nx[0]; w3[1] = nx[1]; w3[2] = nx[2];
        r = rn; g = gn;
        rn += dr; gn += dg;
        if (gn >= groups_per_row) { gn -= groups_per_row; ++rn; }
    }
    if (a.early) grid_dependency_wait();
}

// ---- PTX helpers: mbarrier, TMA tile load, shared-memory loads --------------------------

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
// TMA: one 3-D box {x, y, plane} of the planar crop tensor -> dense [plane][row][col] tile
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void* tmap, int x, int y, int z, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(dst), "l"(tmap), "r"(x), "r"(y), "r"(z), "r"(bar) : "memory");
}
__device__ __forceinline__ uint2 lds_v2(uint32_t a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ NodeT lds_node(uint32_t a) { return lds_v2(a); }
__device__ __forceinline__ uint32_t lds_u16(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ double lds_f64(uint32_t a) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
    return v;
}

// ---- per-label accumulation (np.unique :97 + first loop of compileSaliencyMap :235-238) ----
// d = p1 - (max(sa, thr) - thr) per pixel (:237); per label: sum d, sum |d|, area, bounding
// box.  Runs in K1's epilogue: the 32 lanes of a warp hold 32 consecutive pixels of one
// row; lanes with equal labels are combined with shuffles so that a warp issues one set of
// atomics per distinct label.
struct SegAcc {
    const int32_t* labels;     // [ch*cw]
    int n_labels;
    double thr;                // outlier_threshold
    double* sum;               // [S]
    double* asum;              // [S]
    int* area;                 // [S]
    int* rmin;                 // [S] init INT_MAX
    int* rmax;                 // [S] init -1
    int* cmin;                 // [S] bounding columns of the label (K2's exact path visits only the box)
    int* cmax;
    int* err;                  // STICKY per-handle word: set to 1 on an out-of-range label, cleared by the host once read
};

__device__ __forceinline__ double contribution(double p1, double sa, double thr) {
    return __dsub_rn(p1, __dsub_rn(fmax(sa, thr), thr));
}

// One run of a thread's column: `cnt` pixels of label `lab` in rows [r0, r1] with sum `sm` and
// sum of magnitudes `as`.  lab < 0: the lane does not take part.  Lanes with equal labels are
// combined (shuffles for the float64 sums, redux.sync for the integers) and the group's
// leader issues one set of atomics.
__device__ __forceinline__ void segment_flush(const SegAcc& s, int lab, double sm, double as, int cnt, int r0, int r1, int col) {
    const int lane = threadIdx.x & 31;
    unsigned todo = __ballot_sync(0xffffffffu, lab >= 0);
    while (todo) {
        const int leader = __ffs(todo) - 1;
        const int L = __shfl_sync(0xffffffffu, lab, leader);
        const bool mine = (lab == L);
        const unsigned members = __ballot_sync(0xffffffffu, mine);
        double x = mine ? sm : 0.0, y = mine ? as : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            x += __shfl_xor_sync(0xffffffffu, x, o);
            y += __shfl_xor_sync(0xffffffffu, y, o);
        }
        const int n = __reduce_add_sync(0xffffffffu, mine ? cnt : 0);
        const int lo = __reduce_min_sync(0xffffffffu, mine ? r0 : 0x7fffffff);
        const int hi = __reduce_max_sync(0xffffffffu, mine ? r1 : -1);
        const int cl = __reduce_min_sync(0xffffffffu, mine ? col : 0x7fffffff);
        const int ch = __reduce_max_sync(0xffffffffu, mine ? col : -1);
        if (lane == leader) {
            atomicAdd(s.sum + L, x);
            atomicAdd(s.asum + L, y);
            atomicAdd(s.area + L, n);
            atomicMin(s.rmin + L, lo);
            atomicMax(s.rmax + L, hi);
            atomicMin(s.cmin + L, cl);
            atomicMax(s.cmax + L, ch);
        }
        todo &= ~members;
    }
}

struct ScoreArgs {
    int cw, ch;                      // crop size
    int tiles_x, tiles_y;            // tiles of THIS launch: tile rows [tile_y0, tile_y0 + tiles_y)
    int tile_y0;
    Geom g;
    unsigned* tile_counter;          // dynamic tile scheduler (zeroed by K0)
    DevForest f0, f1;
    TopNodes top0, top1;             // first two levels of f0 / f1 (constant bank)
    int depth;                       // levels walked in every tree: max depth over f0 (and f1)
    int blend;                       // 0/1: f1 (and pca1) valid
    double w0, w1;                   // np.average weights
    int novelty;                     // 0/1
    DevPCA pca0, pca1;               // rank-1 PCAs of the in-line pass (unused when nov_in is set)
    double* p1_out;                  // [ch*cw], or NULL: not kept (only pcm_set_debug keeps the per-pixel maps; K2's exact
    double* sa_out;                  // path recomputes the few pixels it needs).  sa_out: novelty only
    SegAcc seg;                      // per-label accumulators (epilogue)
    const double* nov_in;            // novelty on and a PCA of two or more components: [ch*cw] blended error computed by
                                     // novelty_kernel, which K1 reads instead of running its rank-1 pass; else NULL
};

// One forest over the thread's PIX_PER_THREAD pixels; leaf fractions are added in
// estimator order (sklearn ensemble/_forest.py: all_proba += prediction).
// Branch-free: the PIX_PER_THREAD pointer chases are issued level by level so that
// their dependent shared-memory loads overlap.  SM = forest staged in shared memory
// (node links are absolute shared addresses); otherwise nodes/leaves are read through L1.
// ---- node test -------------------------------------------------------------------------------
// Tile samples are u8 values v, node word x = tap << 16 | thr; right iff v > thr.  (A variant with 2-byte
// samples and one half-precision compare per node -- no mask on the ALU pipe -- was built and measured in
// round 1: no gain, the shared-memory pipe binds; removed in round 2, see profiles/README.md.)
__device__ __forceinline__ bool goes_right(uint32_t v, uint32_t x) { return v > (x & 0xffffu); }

// left + NODE_BYTES (the adjacent right child) iff the sample goes right: one compare + one predicated add
__device__ __forceinline__ uint32_t step_child(uint32_t left, uint32_t v, uint32_t x) {
    asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %2, 0xffff;\n\tsetp.gt.u32 p, %1, t;\n\t@p add.u32 %0, %0, 8;\n\t}"
        : "+r"(left) : "r"(v), "r"(x));
    return left;
}

// DEPTH > 0: every tree of the forest is walked DEPTH levels (compile-time, fully unrolled);
// DEPTH == 0: `depth` levels (kernel-uniform run-time value).  Walking a tree deeper than it is
// costs nothing but time -- leaves self-loop -- so one depth serves the whole forest.
template <bool SM, int DEPTH, int PIX_PER_THREAD>
__device__ __forceinline__ void traverse_forest(const uint32_t nodes_s, const uint32_t leaves_s,
                                                const uint8_t* __restrict__ nodes_g,
                                                const uint8_t* __restrict__ leaves_g,
                                                const int4* __restrict__ trees, const int n_trees, const int depth,
                                                const TopNodes& top,
                                                const uint32_t (&pix)[PIX_PER_THREAD],
                                                double (&acc)[PIX_PER_THREAD]) {
    const uint32_t base = SM ? nodes_s : 0u;
    const uint32_t vdelta = leaves_s - nodes_s;   // shared path: leaf value of the entry at ref = [ref + vdelta]

    auto descend = [&](uint32_t (&ref)[PIX_PER_THREAD], const int levels) {
        auto level = [&]() {
            NodeT nd[PIX_PER_THREAD];
            uint32_t v[PIX_PER_THREAD];
#pragma unroll
            for (int g = 0; g < PIX_PER_THREAD; ++g)
                nd[g] = SM ? lds_node(ref[g]) : __ldg(reinterpret_cast<const NodeT*>(nodes_g + ref[g]));
#pragma unroll
            for (int g = 0; g < PIX_PER_THREAD; ++g) v[g] = lds_u8(pix[g] + node_tap(nd[g]));
#pragma unroll
            for (int g = 0; g < PIX_PER_THREAD; ++g) ref[g] = step_child(node_left(nd[g]), v[g], nd[g].x);
        };
        if (DEPTH > 0) {
#pragma unroll
            for (int l = 0; l < levels; ++l) level();
        } else {
#pragma unroll 1
            for (int l = 0; l < levels; ++l) level();
        }
#pragma unroll
        for (int g = 0; g < PIX_PER_THREAD; ++g) {
            const double leaf = SM ? lds_f64(ref[g] + vdelta)
                                   : __ldg(reinterpret_cast<const double*>(leaves_g + ref[g]));
            acc[g] = __dadd_rn(acc[g], leaf);
        }
    };

    // trees whose first two levels sit in the constant bank (all of them in practice)
    const int n_top = n_trees < MAX_TOP_TREES ? n_trees : MAX_TOP_TREES;
    const int rest = DEPTH > 0 ? (DEPTH > 2 ? DEPTH - 2 : 0) : (depth > 2 ? depth - 2 : 0);
#pragma unroll 1
    for (int t = 0; t < n_top; ++t) {
        // levels 0 and 1 from warp-uniform operands; also right for trees of depth < 2 because a
        // leaf pseudo-node selects itself
        const NodeT e0 = top.n[t][0], eL = top.n[t][1], eR = top.n[t][2];
        uint32_t ref[PIX_PER_THREAD], v[PIX_PER_THREAD], x1[PIX_PER_THREAD];
#pragma unroll
        for (int g = 0; g < PIX_PER_THREAD; ++g) v[g] = lds_u8(pix[g] + node_tap(e0));
#pragma unroll
        for (int g = 0; g < PIX_PER_THREAD; ++g) {
            const bool right = goes_right(v[g], e0.x);
            x1[g] = right ? eR.x : eL.x;   // packed tap | thr of the level-1 node
            ref[g] = (right ? node_left(eR) : node_left(eL)) + base;
        }
#pragma unroll
        for (int g = 0; g < PIX_PER_THREAD; ++g) v[g] = lds_u8(pix[g] + (x1[g] >> 16));
#pragma unroll
        for (int g = 0; g < PIX_PER_THREAD; ++g) ref[g] = step_child(ref[g], v[g], x1[g]);
        descend(ref, DEPTH > 0 ? (DEPTH > 2 ? DEPTH - 2 : 0) : rest);
    }
#pragma unroll 1
    for (int t = n_top; t < n_trees; ++t) {
        uint32_t ref[PIX_PER_THREAD];
#pragma unroll
        for (int g = 0; g < PIX_PER_THREAD; ++g) ref[g] = (uint32_t)trees[t].x + base;
        descend(ref, DEPTH > 0 ? DEPTH : depth);
    }
}

// L1 reconstruction error of a rank-1 PCA over the star features (:58-60):
//   t = sum_f x_f c_f - mean.c ;  err = sum_f |x_f - (t c_f + mean_f)|,  x_f = v_f / 255, v_f = -1 off-crop
// The feature loop runs tap by tap, plane by plane (it = k * NCH + p); comp / comp255 / mean and the tile byte offset
// of every feature are staged in shared memory IN THAT ORDER by the kernel prologue, so the loop body is a broadcast
// load of the three coefficients and, per pixel, one tile byte, one exact u8 -> f64 conversion and the FMAs.  A thread
// whose pixels lie at least n away from every crop edge (`interior`) has no tap outside the crop and skips the
// validity plane altogether.
template <int NCH, int PIX_PER_THREAD>
__device__ __forceinline__ void novelty_error(const double* __restrict__ comp, const double* __restrict__ comp255,
                                              const double* __restrict__ mean, const uint32_t* __restrict__ noff,
                                              const double mdc, const int* __restrict__ sp, const Geom& g, const bool interior,
                                              const uint32_t (&pix)[PIX_PER_THREAD], double (&err)[PIX_PER_THREAD]) {
    // sp[k] and the plane offsets are BYTE offsets
    const int vplane = NCH * g.PS;
    double t[PIX_PER_THREAD];
#pragma unroll
    for (int i = 0; i < PIX_PER_THREAD; ++i) t[i] = 0.0;
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
#pragma unroll 1
        for (int k = 0; k < g.K; ++k) {
            unsigned ok = (1u << PIX_PER_THREAD) - 1u;
            if (!interior) {
                const int so = sp[k];
                ok = 0;
#pragma unroll
                for (int i = 0; i < PIX_PER_THREAD; ++i) ok |= (unsigned)(lds_u8(pix[i] + vplane + so) != 0) << i;
            }
#pragma unroll
            for (int p = 0; p < NCH; ++p) {
                const int it = k * NCH + p;
                const uint32_t off = noff[it];
                if (pass == 0) {
                    const double c255 = comp255[it];
#pragma unroll
                    for (int i = 0; i < PIX_PER_THREAD; ++i) {
                        const double v = ((ok >> i) & 1u) ? u8_to_double(lds_u8(pix[i] + off)) : -1.0;
                        t[i] = fma(v, c255, t[i]);
                    }
                } else {
                    const double c = comp[it], mu = mean[it];
#pragma unroll
                    for (int i = 0; i < PIX_PER_THREAD; ++i) {
                        const double v = ((ok >> i) & 1u) ? u8_to_double(lds_u8(pix[i] + off)) : -1.0;
                        err[i] += fabs(fma(v, 1.0 / 255.0, -fma(t[i], c, mu)));
                    }
                }
            }
        }
        if (pass == 0) {
#pragma unroll
            for (int i = 0; i < PIX_PER_THREAD; ++i) t[i] -= mdc;
        }
    }
}

__device__ __forceinline__ double blend2(double a, double b, double w0, double w1) {
    // np.average([a, b], weights=[w0, w1]) = (a*w0 + b*w1) / (w0 + w1), no contraction
    return __ddiv_rn(__dadd_rn(__dmul_rn(a, w0), __dmul_rn(b, w1)), __dadd_rn(w0, w1));
}

// Tile buffers per CTA: 2 = the TMA load of tile i+1 overlaps the scoring of tile i.
#ifndef PCM_U8_TILE_BUFS
#define PCM_U8_TILE_BUFS 2          // tuning experiments: 1 = single-buffered tiles
#endif
constexpr int N_TILE_BUF = PCM_U8_TILE_BUFS;

struct ScoreSmem {
    uint32_t tiles, bars, sched, sp, f0_nodes, f0_leaves, f0_trees, f1_nodes, f1_leaves, f1_trees, pca0, pca1, nov_off, total;
};

__host__ __device__ inline uint32_t align_up(uint32_t v, uint32_t a) { return (v + a - 1) / a * a; }

// Shared-memory carve-up, identical on host (sizing) and device.
__host__ __device__ inline ScoreSmem score_smem_layout(const Geom& g, const DevForest& f0, const DevForest& f1,
                                                       bool blend, bool novelty, bool forest_smem) {
    ScoreSmem s;
    uint32_t o = 0;
    const int nbuf = N_TILE_BUF;
    s.tiles = o;  o = align_up(o + nbuf * align_up(g.n_planes * g.PS, 128), 128);
    s.bars = o;   o += 8 * nbuf;
    s.sched = o;  o = align_up(o + 4 * nbuf, 16);
    s.sp = o;     o = align_up(o + 4 * g.K, 16);
    s.f0_nodes = s.f0_leaves = s.f1_nodes = s.f1_leaves = 0;
    s.f0_trees = o;  o = align_up(o + 16 * f0.n_trees, 16);
    s.f1_trees = o;
    if (blend) o = align_up(o + 16 * f1.n_trees, 16);
    if (forest_smem) {
        s.f0_nodes = o;  o = align_up(o + NODE_BYTES * f0.n_nodes, 16);
        s.f0_leaves = o; o = align_up(o + 8 * f0.n_nodes, 16);
        if (blend) {
            s.f1_nodes = o;  o = align_up(o + NODE_BYTES * f1.n_nodes, 16);
            s.f1_leaves = o; o = align_up(o + 8 * f1.n_nodes, 16);
        }
    }
    s.pca0 = s.pca1 = s.nov_off = 0;
    if (novelty) {
        s.pca0 = o; o = align_up(o + 24 * g.F, 16);
        if (blend) { s.pca1 = o; o = align_up(o + 24 * g.F, 16); }
        s.nov_off = o; o = align_up(o + 4 * g.F, 16);
    }
    s.total = o;
    return s;
}

template <typename T>
__device__ __forceinline__ void copy_to_smem(T* dst, const T* __restrict__ src, int n) {
    for (int i = threadIdx.x; i < n; i += NTHREADS) dst[i] = src[i];
}

// stage a forest's nodes in shared memory, turning child offsets into absolute shared addresses
__device__ __forceinline__ void stage_nodes(uint8_t* dst, const NodeT* __restrict__ src, int n) {
    const uint32_t base = smem_u32(dst);
    for (int i = threadIdx.x; i < n; i += NTHREADS) {
        NodeT nd = src[i];
        node_set_left(nd, node_left(nd) + base);
        reinterpret_cast<NodeT*>(dst)[i] = nd;
    }
}

// K1 -----------------------------------------------------------------------------
// Persistent CTAs; tiles are handed out by an atomic counter and arrive through a
// two-stage TMA pipeline (the box of tile i+1 is in flight while tile i is scored).
template <bool FOREST_SMEM, int DEPTH, int PIX_PER_THREAD>
__global__ void __launch_bounds__(NTHREADS, PCM_MIN_CTAS) score_kernel(const __grid_constant__ CUtensorMap tmap, const ScoreArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    const Geom& g = a.g;
    const ScoreSmem L = score_smem_layout(g, a.f0, a.f1, a.blend != 0, a.novelty != 0 && !a.nov_in, FOREST_SMEM);
    constexpr int TILE_H = ROW_GROUPS * PIX_PER_THREAD;     // rows per tile; a.tiles_y = ceil(ch / TILE_H)
    const int PH = TILE_H + 2 * g.n;                        // rows of a TMA box (tile + vertical halo)
    const uint32_t tile_bytes = align_up(g.n_planes * g.PS, 128);
    const uint32_t tiles_s = smem_u32(smem + L.tiles);
    const uint32_t bars_s = smem_u32(smem + L.bars);
    volatile int* sched = reinterpret_cast<volatile int*>(smem + L.sched);
    int* sp = reinterpret_cast<int*>(smem + L.sp);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_tiles = a.tiles_x * a.tiles_y;
    const uint32_t box_bytes = (uint32_t)(g.n_planes * g.RS * PH);   // bytes all the boxes of one tile bring

    auto issue = [&](int buf) {   // thread 0: claim the next tile and start its TMA load
        const int t = (int)atomicAdd(a.tile_counter, 1u);
        sched[buf] = t;
        if (t < n_tiles) {
            const uint32_t bar = bars_s + 8 * buf;
            mbar_expect_tx(bar, box_bytes);
            // one {RS, PH, 1} box per plane, each to its fixed plane slot of the buffer
            const int x = (t % a.tiles_x) * TILE_W - g.HX, y = (a.tile_y0 + t / a.tiles_x) * TILE_H - g.n;
            for (int pl = 0; pl < g.n_planes; ++pl)
                tma_load_3d(tiles_s + buf * tile_bytes + pl * g.PS, &tmap, x, y, pl, bar);
        }
    };

    // ---- once per CTA: tap offsets, forests, PCA vectors -> smem.  None of it depends on the
    //      preceding kernel (K0), so under programmatic dependent launch it overlaps K0's tail ----
    for (int k = tid; k < g.K; k += NTHREADS) {
        int dr, dc;
        star_tap(k, dr, dc);
        sp[k] = (dr + g.n) * g.RS + (dc + g.HX);
    }
    copy_to_smem(reinterpret_cast<int4*>(smem + L.f0_trees), a.f0.trees, a.f0.n_trees);
    if (a.blend) copy_to_smem(reinterpret_cast<int4*>(smem + L.f1_trees), a.f1.trees, a.f1.n_trees);
    const int4* f0t = reinterpret_cast<const int4*>(smem + L.f0_trees);
    const int4* f1t = reinterpret_cast<const int4*>(smem + L.f1_trees);
    if (FOREST_SMEM) {
        stage_nodes(smem + L.f0_nodes, a.f0.nodes, a.f0.n_nodes);
        copy_to_smem(reinterpret_cast<double*>(smem + L.f0_leaves), a.f0.leaves, a.f0.n_nodes);
        if (a.blend) {
            stage_nodes(smem + L.f1_nodes, a.f1.nodes, a.f1.n_nodes);
            copy_to_smem(reinterpret_cast<double*>(smem + L.f1_leaves), a.f1.leaves, a.f1.n_nodes);
        }
    }
    // PCA vectors in the ORDER the novelty loop walks the features (tap by tap, plane by plane): entry it = k * nch + p
    // holds feature f = (p / 3) * 3K + 3k + p % 3 (:272), next to the feature's byte offset inside the tile
    const double *p0c = nullptr, *p0c255 = nullptr, *p0m = nullptr, *p1c = nullptr, *p1c255 = nullptr, *p1m = nullptr;
    const uint32_t* noff = reinterpret_cast<const uint32_t*>(smem + L.nov_off);
    if (a.novelty && !a.nov_in) {
        const int nch = 3 * g.n_spaces;
        double* d0 = reinterpret_cast<double*>(smem + L.pca0);
        double* d1 = reinterpret_cast<double*>(smem + L.pca1);
        uint32_t* no = reinterpret_cast<uint32_t*>(smem + L.nov_off);
        for (int it = tid; it < g.F; it += NTHREADS) {
            const int k = it / nch, p = it - k * nch;
            const int f = (p / 3) * 3 * g.K + 3 * k + (p % 3);
            int dr, dc;
            star_tap(k, dr, dc);
            no[it] = (uint32_t)(p * g.PS + (dr + g.n) * g.RS + (dc + g.HX));
            d0[it] = a.pca0.comp[f]; d0[g.F + it] = a.pca0.comp255[f]; d0[2 * g.F + it] = a.pca0.mean[f];
            if (a.blend) { d1[it] = a.pca1.comp[f]; d1[g.F + it] = a.pca1.comp255[f]; d1[2 * g.F + it] = a.pca1.mean[f]; }
        }
        p0c = d0; p0c255 = d0 + g.F; p0m = d0 + 2 * g.F;
        p1c = d1; p1c255 = d1 + g.F; p1m = d1 + 2 * g.F;
    }
    grid_dependency_wait();     // K0's planes, tile counter and per-label resets are complete and visible
    grid_launch_dependents();
    if (tid == 0) {
        for (int b = 0; b < N_TILE_BUF; ++b) mbar_init(bars_s + 8 * b, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        if (N_TILE_BUF > 1) issue(0);
    }

    __syncthreads();

    const uint32_t f0n_s = smem_u32(smem + L.f0_nodes), f0l_s = smem_u32(smem + L.f0_leaves);
    const uint32_t f1n_s = smem_u32(smem + L.f1_nodes), f1l_s = smem_u32(smem + L.f1_leaves);
    const uint8_t* f0n_g = reinterpret_cast<const uint8_t*>(a.f0.nodes);
    const uint8_t* f0l_g = reinterpret_cast<const uint8_t*>(a.f0.leaves);
    const uint8_t* f1n_g = reinterpret_cast<const uint8_t*>(a.f1.nodes);
    const uint8_t* f1l_g = reinterpret_cast<const uint8_t*>(a.f1.leaves);

    const int col = (warp & 1) * 32 + lane;
    const int row0 = (warp >> 1) * PIX_PER_THREAD;
    uint32_t phase = 0;   // bit b = parity to wait for on buffer b
    for (int buf = 0;; buf = (N_TILE_BUF > 1) ? (buf ^ 1) : 0) {
        if (N_TILE_BUF == 1) {
            if (tid == 0) issue(0);
            __syncthreads();
        }
        const int tile = sched[buf];
        if (tile >= n_tiles) break;
        if (N_TILE_BUF > 1 && tid == 0) issue(buf ^ 1);   // buffer buf^1 was released by the barrier below
        mbar_wait(bars_s + 8 * buf, (phase >> buf) & 1u);
        phase ^= 1u << buf;

        const int tx0 = (tile % a.tiles_x) * TILE_W, ty0 = (a.tile_y0 + tile / a.tiles_x) * TILE_H;
        const int ox = tx0 + col;
        uint32_t pix[PIX_PER_THREAD];
#pragma unroll
        for (int i = 0; i < PIX_PER_THREAD; ++i) pix[i] = tiles_s + buf * tile_bytes + (row0 + i) * g.RS + col;

        // labels of the thread's pixels: requested now, consumed in the epilogue (their HBM/L2
        // latency hides behind the forest traversal)
        int lab[PIX_PER_THREAD];
#pragma unroll
        for (int i = 0; i < PIX_PER_THREAD; ++i) {
            const int oy = ty0 + row0 + i;
            lab[i] = (ox < a.cw && oy < a.ch) ? __ldg(a.seg.labels + (size_t)oy * a.cw + ox) : -1;
        }

        double p[PIX_PER_THREAD];
#pragma unroll
        for (int i = 0; i < PIX_PER_THREAD; ++i) p[i] = 0.0;
        traverse_forest<FOREST_SMEM, DEPTH, PIX_PER_THREAD>(f0n_s, f0l_s, f0n_g, f0l_g, f0t, a.f0.n_trees, a.depth, a.top0, pix, p);
        const double T0 = (double)a.f0.n_trees;
#pragma unroll
        for (int i = 0; i < PIX_PER_THREAD; ++i) p[i] = __ddiv_rn(p[i], T0);
        if (a.blend) {
            double q[PIX_PER_THREAD];
#pragma unroll
            for (int i = 0; i < PIX_PER_THREAD; ++i) q[i] = 0.0;
            traverse_forest<FOREST_SMEM, DEPTH, PIX_PER_THREAD>(f1n_s, f1l_s, f1n_g, f1l_g, f1t, a.f1.n_trees, a.depth, a.top1, pix, q);
            const double T1 = (double)a.f1.n_trees;
#pragma unroll
            for (int i = 0; i < PIX_PER_THREAD; ++i) p[i] = blend2(p[i], __ddiv_rn(q[i], T1), a.w0, a.w1);
        }
        double e[PIX_PER_THREAD];
#pragma unroll
        for (int i = 0; i < PIX_PER_THREAD; ++i) e[i] = 0.0;
        if (a.novelty && a.nov_in) {
#pragma unroll
            for (int i = 0; i < PIX_PER_THREAD; ++i) {
                const int oy = ty0 + row0 + i;
                if (ox < a.cw && oy < a.ch) e[i] = __ldg(a.nov_in + (size_t)oy * a.cw + ox);
            }
        } else if (a.novelty) {
            // no tap of this thread's pixels can fall outside the crop: the validity plane need not be read
            const bool interior = ox >= g.n && ox + g.n < a.cw && ty0 + row0 >= g.n && ty0 + row0 + PIX_PER_THREAD - 1 + g.n < a.ch;
            auto run = [&](const double* c, const double* c255, const double* mu, double mdc, double (&out)[PIX_PER_THREAD]) {
                switch (g.n_spaces) {
                    case 1: novelty_error<3, PIX_PER_THREAD>(c, c255, mu, noff, mdc, sp, g, interior, pix, out); break;
                    case 2: novelty_error<6, PIX_PER_THREAD>(c, c255, mu, noff, mdc, sp, g, interior, pix, out); break;
                    default: novelty_error<9, PIX_PER_THREAD>(c, c255, mu, noff, mdc, sp, g, interior, pix, out); break;
                }
            };
            run(p0c, p0c255, p0m, a.pca0.mean_dot_comp, e);
            if (a.blend) {
                double e1[PIX_PER_THREAD];
#pragma unroll
                for (int i = 0; i < PIX_PER_THREAD; ++i) e1[i] = 0.0;
                run(p1c, p1c255, p1m, a.pca1.mean_dot_comp, e1);
#pragma unroll
                for (int i = 0; i < PIX_PER_THREAD; ++i) e[i] = blend2(e[i], e1[i], a.w0, a.w1);
            }
        }
        // ---- epilogue: P(fg) [, err] to HBM and the per-label sums (K2 fused here) --------------
        // A thread walks down its column and merges consecutive pixels of the same label; the
        // warp flushes (segment_flush) only when some lane's label changes, so a superpixel that
        // spans the thread's rows costs one flush per tile instead of one per row.
        int run_lab = -1, run_cnt = 0, run_r0 = 0, run_r1 = 0;
        double run_sum = 0.0, run_abs = 0.0;
#pragma unroll
        for (int i = 0; i < PIX_PER_THREAD; ++i) {
            const int oy = ty0 + row0 + i;
            int l = lab[i];
            if (ox < a.cw && oy < a.ch) {
                const size_t o = (size_t)oy * a.cw + ox;
                if (a.p1_out) {
                    a.p1_out[o] = p[i];
                    if (a.novelty && !a.nov_in) a.sa_out[o] = e[i];
                }
                if (l < 0 || l >= a.seg.n_labels) { *a.seg.err = 1; l = -1; }
            }
            const bool change = (l != run_lab) && run_lab >= 0;
            if (__any_sync(0xffffffffu, change)) {
                segment_flush(a.seg, change ? run_lab : -1, run_sum, run_abs, run_cnt, run_r0, run_r1, ox);
                if (change) run_lab = -1;
            }
            if (l >= 0) {
                const double d = contribution(p[i], e[i], a.seg.thr);
                if (run_lab < 0) { run_lab = l; run_cnt = 0; run_sum = 0.0; run_abs = 0.0; run_r0 = oy; }
                run_sum += d; run_abs += fabs(d); run_cnt++; run_r1 = oy;
            }
        }
        segment_flush(a.seg, run_lab, run_sum, run_abs, run_cnt, run_r0, run_r1, ox);
        __syncthreads();   // tile buffer `buf` may be refilled; sched[buf^1] is visible
    }
}

}  // namespace pcm
