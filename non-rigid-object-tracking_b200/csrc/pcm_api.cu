// pcm_api.cu -- host side of libpcm_b200.so: the C ABI declared in include/pcm_b200.h.
//
// Owns device memory, streams, the packed forests, and launches the kernels of
// pcm_kernels.cuh.  No CPU implementation of the hot path exists in this library:
// every entry point either runs the CUDA kernels or fails.
#include "../../include/pcm_b200.h"
#include "pcm_kernels.cuh"
#include "pcm_score_variants.h"
#include "pcm_quickshift.cuh"
#include "pcm_forest_fit.cuh"
#include "pcm_prior.cuh"
#include "pcm_slic.cuh"
#include "pcm_host.h"

#include <cudaTypedefs.h>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <string>
#include <utility>
#include <vector>

using namespace pcm;

namespace pcm {   // pcm_host_simd.cpp
void gather_strided(const uint8_t* src, int64_t stride, uint8_t* dst, int n);
void scatter_strided(const uint8_t* src, uint8_t* dst, int64_t stride, int n);
// pcm_felzenszwalb.cpp
int felzenszwalb(const uint8_t* frame, int64_t stride, int cx, int cy, int w, int h, double scale, double sigma,
                 int min_size, const double* kernel, int radius, int32_t* labels_out);
int felzenszwalb_graph(int n_vertices, int n_edges, const int32_t* a, const int32_t* b, const double* cost, double scale,
                       int min_size, int32_t* labels_out);
// pcm_slic.cpp
int slic(const uint8_t* frame, int64_t stride, int cx, int cy, int w, int h, int n_segments, double compactness, double sigma,
         const double* kernel, int radius, int max_iter, int start_label, int32_t* labels_out);
}

// ---------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------
static thread_local std::string g_last_error;

static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

#define CUDA_TRY(expr)                                                                       \
    do {                                                                                     \
        cudaError_t e__ = (expr);                                                            \
        if (e__ != cudaSuccess)                                                              \
            return fail(PCM_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                        __FILE__, __LINE__);                                                 \
    } while (0)

// ---------------------------------------------------------------------------------
// PCM_TRACE=1: wall-clock breakdown of the host-buffer entry points, printed at pcm_destroy
// ---------------------------------------------------------------------------------
#include <chrono>
static bool trace_enabled() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("PCM_TRACE"); v = (e && e[0] == '1') ? 1 : 0; }
    return v == 1;
}
struct HostTrace {
    enum { UPD_SYNC, UPD_STAGE, UPD_ENQUEUE, UPD_WAIT, UPD_D2H, UPD_SCATTER, IOU_STAGE, IOU_WAIT, N };
    double ms[N] = {0};
    long calls[N] = {0};
    std::chrono::steady_clock::time_point t;
    void start() { if (trace_enabled()) t = std::chrono::steady_clock::now(); }
    long seen[N] = {0};
    void lap(int id) {
        if (!trace_enabled()) return;
        auto now = std::chrono::steady_clock::now();
        if (++seen[id] > 8) {                 // the first calls allocate (pinned memory, events): not what is being traced
            ms[id] += std::chrono::duration<double, std::milli>(now - t).count();
            calls[id]++;
        }
        t = now;
    }
    void report() const {
        if (!trace_enabled()) return;
        static const char* names[N] = {"update: reserve+sync", "update: stage+H2D issue", "update: enqueue kernels",
                                       "update: wait (H2D, kernels, first D2H band)", "update: wait for later D2H bands", "update: scatter mask",
                                       "iou: verify mask / stage+H2D issue",
                                       "iou: kernel+D2H wait"};
        for (int i = 0; i < N; ++i) {                   // laps that occur several times per call are summed per call
            const long per = calls[i < IOU_STAGE ? UPD_SYNC : IOU_WAIT];
            if (calls[i] && per) fprintf(stderr, "[pcm trace] %-46s %8.3f ms/call over %ld calls\n", names[i], ms[i] / per, per);
        }
    }
};

// ---------------------------------------------------------------------------------
// grow-only buffers
// ---------------------------------------------------------------------------------
// Blocks released by a handle are parked in a process-wide cache and handed to the next handle
// that asks for that much memory: a sweep creates and destroys one handle per sequence, and
// cudaFree / cudaFreeHost / cudaMallocHost cost far more than a whole short sequence.
#include <mutex>
class BlockCache {
public:
    static BlockCache& instance() { static BlockCache c; return c; }
    // smallest parked block of `device` (or pinned: device = -1) with capacity in [bytes, 4 * bytes]
    bool take(int device, size_t bytes, void** p, size_t* cap) {
        std::lock_guard<std::mutex> lk(m_);
        int best = -1;
        for (int i = 0; i < (int)blocks_.size(); ++i) {
            const Block& b = blocks_[i];
            if (b.device == device && b.cap >= bytes && b.cap <= 4 * bytes + (1u << 16) &&
                (best < 0 || b.cap < blocks_[best].cap))
                best = i;
        }
        if (best < 0) return false;
        *p = blocks_[best].p;
        *cap = blocks_[best].cap;
        total_[device < 0] -= blocks_[best].cap;
        blocks_.erase(blocks_.begin() + best);
        return true;
    }
    // returns false when the cache is full and the caller has to free the block itself
    bool park(int device, void* p, size_t cap) {
        std::lock_guard<std::mutex> lk(m_);
        // (a sweep closes dozens of handles at once, the fitting ones with ~100 MB each; a block that does not fit here is
        // cudaFree'd, which waits for the whole device)
        const size_t limit = device < 0 ? ((size_t)4 << 30) : ((size_t)32 << 30);
        if (total_[device < 0] + cap > limit || blocks_.size() >= 4096) return false;
        blocks_.push_back({device, p, cap});
        total_[device < 0] += cap;
        return true;
    }
private:
    struct Block { int device; void* p; size_t cap; };
    std::mutex m_;
    std::vector<Block> blocks_;
    size_t total_[2] = {0, 0};
};

// DevBuf / PinBuf own their block: it goes back to the BlockCache (or is freed) when the buffer is destroyed.  A move
// hands the block over, at the same address, and leaves the source empty.
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int device = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)), device(o.device) {}
    ~DevBuf() { release(); }
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        // growing: kernels queued by an asynchronous entry point may still use the old block, and a
        // parked block can be handed to another handle at once -- wait for the device first (rare)
        if (p) cudaDeviceSynchronize();
        release();
        cudaGetDevice(&device);
        if (BlockCache::instance().take(device, bytes, &p, &cap)) return cudaSuccess;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        else p = nullptr;
        return e;
    }
    void release() {
        if (p && !BlockCache::instance().park(device, p, cap)) cudaFree(p);
        p = nullptr; cap = 0;
    }
    template <typename T> T* as() const { return static_cast<T*>(p); }
};

struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    PinBuf() = default;
    PinBuf(const PinBuf&) = delete;
    PinBuf& operator=(const PinBuf&) = delete;
    PinBuf(PinBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    ~PinBuf() { release(); }
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        release();
        if (BlockCache::instance().take(-1, bytes, &p, &cap)) return cudaSuccess;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e == cudaSuccess) cap = want;
        else p = nullptr;
        return e;
    }
    void release() {
        if (p && !BlockCache::instance().park(-1, p, cap)) cudaFreeHost(p);
        p = nullptr; cap = 0;
    }
    template <typename T> T* as() const { return static_cast<T*>(p); }
};

// ---------------------------------------------------------------------------------
// caller-registered (page-locked) host ranges: pcm_host_register / pcm_host_unregister.
// A frame / truth image that lies inside one is copied to the device straight from the caller's
// memory; everything else is staged through the handle's pinned buffers.
// ---------------------------------------------------------------------------------
class HostRegistry {
public:
    static HostRegistry& instance() { static HostRegistry r; return r; }
    bool contains(const void* p, size_t bytes) {
        const uintptr_t lo = reinterpret_cast<uintptr_t>(p), hi = lo + bytes;
        std::lock_guard<std::mutex> lk(m_);
        for (const R& r : v_)
            if (lo >= r.lo && hi <= r.hi) return true;
        return false;
    }
    void add(const void* p, size_t bytes) {
        std::lock_guard<std::mutex> lk(m_);
        v_.push_back({reinterpret_cast<uintptr_t>(p), reinterpret_cast<uintptr_t>(p) + bytes});
    }
    bool remove(const void* p) {
        std::lock_guard<std::mutex> lk(m_);
        for (size_t i = 0; i < v_.size(); ++i)
            if (v_[i].lo == reinterpret_cast<uintptr_t>(p)) { v_.erase(v_.begin() + i); return true; }
        return false;
    }
private:
    struct R { uintptr_t lo, hi; };
    std::mutex m_;
    std::vector<R> v_;
};

// ---------------------------------------------------------------------------------
// models
// ---------------------------------------------------------------------------------
struct Model {
    int n_frame = 0;
    DevForest forest{};
    DevBuf blob;                  // nodes | leaves | trees, one block (from the process-wide block cache)
    TopNodes top{};               // root + its children of the first MAX_TOP_TREES trees
    bool has_pca = false;
    int pca_k = 0;                // n_components of the PCA
    DevPCA pca{};                 // rank 1: K1's in-line pass
    DevBuf pca_buf;               // comp | comp255 | mean, 3F doubles (rank 1)
    DevBuf pcak_buf;              // novelty_kernel's coefficients: [F][pca_k + 1] in its visiting order (any rank)
    double pcak_mdc[MAX_PCA_K] = {0};   // mean_ . components_[j]
    int max_depth = 0;
};

struct pcm_handle {
    int device = 0;
    int sm_count = 0;
    int max_smem_optin = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    ColorTables* d_tables = nullptr;
    ColorTables h_tables;
    DevBuf err_buf;
    int* d_err = nullptr;         // sticky "label out of range" word: set by K1, cleared by the host once reported
    // true while the last thing this handle queued on its PRIVATE stream is its own K3 / K5: only then may
    // the next K0 start before its predecessor has finished (PlanesArgs::early)
    bool chain_tail = false;
    PFN_cuTensorMapEncodeTiled_v12000 encode_tiled = nullptr;   // driver entry point (no libcuda link)
    bool features_set = false;
    Geom geom{};
    std::vector<Model> models;
    int64_t launches = 0;
    std::atomic<int64_t> bytes_h2d{0}, bytes_d2h{0};   // bytes moved by the host-buffer entry points

    // optional per-kernel event timing
    bool profiling = false;
    struct Timed { int id; cudaEvent_t a, b; };
    std::vector<Timed> pending;
    std::vector<cudaEvent_t> free_events;
    double prof_ms[PCM_NUM_KERNELS] = {0};
    int64_t prof_n[PCM_NUM_KERNELS] = {0};

    // per-update scratch (device)
    DevBuf frame, labels, priors, planes, sched, p1, sa, seg, rmin, rmax, cmin, cmax, decision, scores, flagged, mask, pre, counts;
    // pinned staging (host)
    PinBuf h_frame, h_labels, h_priors, h_mask, h_small;

    // host-path label cache: h_labels / labels hold the label map of the previous pcm_update
    // (label_cache_px elements, 1 MiB chunks); a chunk whose bytes are unchanged is not re-sent
    size_t label_cache_px = 0;
    std::vector<int> label_chunk_max;
    bool label_cache_on = true;   // pcm_set_label_cache

    // over-segmentation on the GPU (quickshift, SLIC): the label map of the last call, and the handoff to pcm_update with
    // labels == NULL, armed by pcm_quickshift / pcm_slic_gpu: the crop `rect` of the host frame `frame` is in `frame` (the
    // device buffer above) and its map of n_labels segments in seg_labels
    DevBuf seg_labels;
    struct {
        bool valid;
        const uint8_t* frame;
        int rect[4];
        int n_labels;
    } handoff = {false, nullptr, {0, 0, 0, 0}, 0};

    // quickshift (pcm_quickshift*): scratch; the noise of the last call with noise and its crop size
    DevBuf qs_lab, qs_dens, qs_noise, qs_parent, qs_root, qs_flag, qs_rank, qs_sums, qs_lin, qs_count;
    PinBuf h_noise;
    int qs_noise_cw = 0, qs_noise_ch = 0;

    // SLIC (pcm_slic_gpu / pcm_slic_device*): scratch.  sl_smooth, sl_img and sl_nearest keep the stage results of the last
    // call (pcm_slic_debug_last).
    DevBuf sl_kernel, sl_smooth, sl_tmp, sl_img, sl_centers, sl_dmin, sl_best, sl_nearest, sl_keys, sl_iota, sl_sidx, sl_begin,
           sl_end, sl_cub, sl_count;
    DevBuf sl_parent, sl_root, sl_csize, sl_piece, sl_psize, sl_off, sl_queue, sl_seen, sl_adj, sl_nxt, sl_val, sl_labels;
    PinBuf h_slic;                // Gaussian weights + seed centres
    int sl_w = 0, sl_h = 0;       // crop of the stage results; 0: none
    // forest training (pcm_fit_forest): feature-major rows resident between calls, scratch, outputs
    DevBuf fit_x, fit_xt, fit_y, fit_counts, fit_rand, fit_samples, fit_tmp, fit_out;
    DevBuf prior_scratch;         // pcm_prior_device: per-keypoint match records
    long long fit_rows_id = 0;
    int fit_n = 0, fit_F = 0;

    // host-path mask mirror: `mask` (device) and `h_mask` (pinned) are dense mir_H x mir_W planes that follow the
    // caller's mask image.  pcm_update writes its crop into both; pcm_iou compares the caller's bytes with the pinned
    // copy band by band (mir_band_rows rows each) and uploads only the bands that differ (or were never synchronised:
    // mir_ok[b] == 0), so the mask pcm_update has just produced is not sent back to the device.
    int mir_H = 0, mir_W = 0, mir_band_rows = 0;
    std::vector<uint8_t> mir_ok;
    cudaEvent_t band_events[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    std::vector<cudaEvent_t> ahead_events;   // pcm_run_frames: frames in flight
    cudaStream_t copy_stream = nullptr;   // host path: row bands of a page-locked caller frame travel here (BandFeed)
    cudaEvent_t feed_events[4] = {nullptr, nullptr, nullptr, nullptr};
    int resident_labels = 0;      // n_labels of the label map the last host pcm_update left on the device (0: none)
    int resident_cw = 0, resident_ch = 0;

    // description of the last update (for pcm_debug_last)
    int last_cw = 0, last_ch = 0, last_S = 0;
    bool last_novelty = false;
    bool last_valid = false;
    bool last_pre = false;
    bool last_maps = false;       // the last update kept its P(fg) / novelty maps
    bool keep_pre = false;        // pcm_set_debug bit 0: K3 also writes the pre-dilation map, K1 the per-pixel P(fg) / novelty maps
    bool force_exact = false;     // pcm_set_debug bit 1: every label takes K2's exact path (tests)
    HostTrace trace;
};

// seg buffer layout: [sum S f64][asum S f64][area S i32][n_flagged i32]
struct SegLayout {
    size_t sum, asum, area, nflag, total;
};
static SegLayout seg_layout(int S) {
    SegLayout l;
    l.sum = 0;
    l.asum = l.sum + sizeof(double) * (size_t)S;
    l.area = l.asum + sizeof(double) * (size_t)S;
    l.nflag = l.area + sizeof(int) * (size_t)S;
    l.nflag = (l.nflag + 7) / 8 * 8;
    l.total = l.nflag + 2 * sizeof(int);
    return l;
}

// PCM_DEBUG_SYNC=1: synchronise after every launch so that a device fault is
// attributed to the kernel that caused it.
static bool debug_sync_enabled() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("PCM_DEBUG_SYNC"); v = (e && e[0] == '1') ? 1 : 0; }
    return v == 1;
}
#define CHECK_LAUNCH(h, name)                                                                   \
    do {                                                                                        \
        CUDA_TRY(cudaGetLastError());                                                           \
        (h)->launches++;                                                                        \
        if (debug_sync_enabled()) {                                                             \
            cudaError_t e2__ = cudaStreamSynchronize((h)->stream);                              \
            if (e2__ != cudaSuccess)                                                            \
                return fail(PCM_E_CUDA, "kernel %s faulted: %s", name, cudaGetErrorString(e2__)); \
        }                                                                                       \
    } while (0)

// ---------------------------------------------------------------------------------
// Programmatic dependent launch: the five kernels of a frame run back to back on one stream.
// Launched with this attribute a kernel's CTAs may become resident while the previous kernel
// drains; each kernel executes `griddepcontrol.wait` (grid_dependency_wait) before it touches
// anything its predecessor wrote -- K1 only after it has staged its forests -- so the launch
// latency and K1's prologue overlap the predecessor's tail.  PCM_PDL=0 switches it off.
// ---------------------------------------------------------------------------------
static bool pdl_enabled() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("PCM_PDL"); v = (e && e[0] == '0') ? 0 : 1; }
    return v == 1;
}
template <typename... KArgs, typename... Args>
static cudaError_t launch_chain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// ---------------------------------------------------------------------------------
// per-kernel timing
// ---------------------------------------------------------------------------------
struct KernelTimer {
    pcm_handle* h;
    int id;
    cudaEvent_t a = nullptr, b = nullptr;
    static cudaEvent_t get(pcm_handle* h) {
        if (!h->free_events.empty()) { cudaEvent_t e = h->free_events.back(); h->free_events.pop_back(); return e; }
        cudaEvent_t e = nullptr;
        cudaEventCreate(&e);
        return e;
    }
    KernelTimer(pcm_handle* h_, int id_) : h(h_), id(id_) {
        if (!h->profiling) return;
        a = get(h); b = get(h);
        cudaEventRecord(a, h->stream);
    }
    ~KernelTimer() {
        if (!a) return;
        cudaEventRecord(b, h->stream);
        h->pending.push_back({id, a, b});
    }
};

// one kernel of the frame chain on the handle's stream: timed under profile id `id`, checked like CHECK_LAUNCH
template <typename... KArgs, typename... Args>
static int launch_timed(pcm_handle* h, int id, const char* name, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                        Args&&... args) {
    {
        KernelTimer kt(h, id);
        CUDA_TRY(launch_chain(kernel, grid, block, smem, h->stream, std::forward<Args>(args)...));
    }
    CHECK_LAUNCH(h, name);
    return PCM_OK;
}

// ---------------------------------------------------------------------------------
// tables (OpenCV's fixed-point LUTs; SURVEY.md §8 a-1, a-2)
// ---------------------------------------------------------------------------------
static void build_tables(ColorTables& t) {
    memset(&t, 0, sizeof t);
    for (int i = 0; i < 256; ++i) {
        double x = i / 255.0;
        double lin = x <= 0.04045 ? x / 12.92 : pow((x + 0.055) / 1.055, 2.4);
        t.gamma[i] = (uint16_t)nearbyint(lin * 2040.0);
    }
    for (int i = 0; i < LAB_CBRT_SIZE; ++i) {
        double x = i / 2040.0;
        double f = x < 216.0 / 24389.0 ? x * (841.0 / 108.0) + 16.0 / 116.0 : cbrt(x);
        t.cbrt_tab[i] = (uint16_t)nearbyint(f * 32768.0);
    }
    // OpenCV evaluates the table with softfloat; float64 differs in exactly these entries
    t.cbrt_tab[49] = 9454;
    t.cbrt_tab[628] = 22126;
    t.sdiv[0] = t.hdiv[0] = 0;
    for (int i = 1; i < 256; ++i) {
        t.sdiv[i] = (int32_t)nearbyint((255 << 12) / (double)i);
        t.hdiv[i] = (int32_t)nearbyint((180 << 12) / (6.0 * i));
    }
}

// ---------------------------------------------------------------------------------
// geometry
// ---------------------------------------------------------------------------------
static Geom make_geom(int n, int n_spaces, const int* ids) {
    Geom g{};
    g.n = n;
    g.n_spaces = n_spaces;
    for (int i = 0; i < n_spaces; ++i) g.space_id[i] = ids[i];
    g.K = 1 + 8 * n;
    g.F = 3 * g.K * n_spaces;
    g.n_planes = 3 * n_spaces + 1;
    g.HX = 16;
    g.RS = TILE_W + 2 * g.HX;
    g.PS = (g.RS * (MAX_TILE_H + 2 * n) + 127) / 128 * 128;     // every plane slot starts on a 128-byte boundary (TMA)
    return g;
}

// ---------------------------------------------------------------------------------
// forest encoding
// ---------------------------------------------------------------------------------
// Largest integer t in [-2, 255] with  float32(v / 255) <= thr  <=>  v <= t  for v in -1..255
// (features are X/255 cast to float32 by sklearn; SURVEY.md §8 a-5).
static int int_threshold(double thr) {
    // f32(v / 255) is increasing in v: start from the real-valued solution and correct by at most a few steps
    auto le = [&](int v) { return (double)(float)((double)v / 255.0) <= thr; };
    if (!(thr >= -1.0)) return le(-1) ? -1 : -2;            // also NaN: nothing passes
    int t = thr >= 1.5 ? 255 : (int)floor(thr * 255.0);
    t = std::min(std::max(t, -2), 255);
    while (t < 255 && le(t + 1)) ++t;
    while (t >= -1 && !le(t)) --t;
    return t;
}

struct EncTree {
    std::vector<NodeT> nodes;     // entries (see pcm_kernels.cuh): left = entry INDEX of the left child here
    std::vector<double> values;   // parallel: class-1 fraction of leaf entries
    int n_leaf = 0;
    int depth = 0;
};

struct Encoder {
    const Geom& g;
    const int32_t* feature;
    const double* threshold;
    const int32_t* left;
    const int32_t* right;
    const double* value1;
    int n;                       // nodes in this tree
    std::vector<int> tint;       // integer threshold per node
    EncTree out;
    std::string err;

    // skip nodes that send every value right (t == -2): they are not representable
    // with an unsigned compare and never needed
    int skip(int i) const {
        while (left[i] != -1 && tint[i] < -1) i = right[i];
        return i;
    }
    bool run() {
        tint.assign(n, 0);
        for (int i = 0; i < n; ++i) {
            if (left[i] == -1) continue;
            if (left[i] < 0 || left[i] >= n || right[i] < 0 || right[i] >= n) { err = "child index out of range"; return false; }
            if (feature[i] < 0 || feature[i] >= g.F) { err = "feature index out of range"; return false; }
            tint[i] = int_threshold(threshold[i]);
        }
        // breadth-first: the root is entry 0, the two children of a node are adjacent entries
        struct Item { int node, entry, depth; };
        std::vector<Item> queue;
        queue.push_back({skip(0), 0, 0});
        out.nodes.assign(1, make_node(0, 0, 0));
        out.values.assign(1, 0.0);
        const int vplane = 3 * g.n_spaces;
        size_t visited = 0;
        for (size_t qi = 0; qi < queue.size(); ++qi) {
            const Item it = queue[qi];
            if (++visited > (size_t)n + 1) { err = "tree is not a tree"; return false; }
            const int i = it.node;
            if (left[i] == -1) {
                out.nodes[it.entry] = make_node(0u, LEAF_THR, (unsigned)it.entry);
                out.values[it.entry] = value1[i];
                out.n_leaf++;
                out.depth = std::max(out.depth, it.depth);
                continue;
            }
            const int f = feature[i];
            const int q = f / (3 * g.K), rem = f % (3 * g.K), k = rem / 3, ch = rem % 3;
            int dr, dc;
            star_tap(k, dr, dc);
            int plane = 3 * q + ch;
            int thr = tint[i];
            if (thr == -1) { plane = vplane; thr = 0; }   // "tap is outside the crop"
            const unsigned off = (unsigned)(plane * g.PS + (dr + g.n) * g.RS + (dc + g.HX));
            if (off >= (1u << 16)) { err = "tap offset overflow"; return false; }
            const int child = (int)out.nodes.size();
            out.nodes.resize(child + 2, make_node(0, 0, 0));
            out.values.resize(child + 2, 0.0);
            out.nodes[it.entry] = make_node(off, (unsigned)thr, (unsigned)child);
            queue.push_back({skip(left[i]), child, it.depth + 1});
            queue.push_back({skip(right[i]), child + 1, it.depth + 1});
        }
        return true;
    }
};

// ---------------------------------------------------------------------------------
// API: lifetime
// ---------------------------------------------------------------------------------
// K1 instantiations (pcm_score_variants.h): forest in shared memory or behind L1, walk depth fixed at compile
// time for the depths the reference's configs use (config.yaml:26 -> 5; benchmark.py:44 -> 7, 10) or taken
// from the arguments (DEPTH = 0), tile height 24 / 28 / 32 rows.
constexpr int N_SCORE_VARIANTS = 3 * N_SCORE_VARIANTS_PER_PPT;
static const ScoreVariant& score_variant(int i) {
    const ScoreVariant* t = i < N_SCORE_VARIANTS_PER_PPT ? score_variants_ppt6()
                          : i < 2 * N_SCORE_VARIANTS_PER_PPT ? score_variants_ppt7() : score_variants_ppt8();
    return t[i % N_SCORE_VARIANTS_PER_PPT];
}
static const ScoreVariant& pick_score_variant(bool smem, int depth, int ppt) {
    int dyn = -1;
    for (int i = 0; i < N_SCORE_VARIANTS; ++i) {
        const ScoreVariant& v = score_variant(i);
        if (v.smem != smem || v.ppt != ppt) continue;
        if (v.depth == depth) return v;
        if (v.depth == 0) dyn = i;
    }
    return score_variant(dyn);
}

// pca_residual_kernel for k = 1..PCM_MAX_PCA_COMPONENTS components, indexed by k - 1; defined right after pcm_create
typedef void (*ResidualFn)(const int16_t*, long long, int, int, const double*, const double*, double*);
namespace { extern const ResidualFn pca_residual_kernels[PCM_MAX_PCA_COMPONENTS]; }

// per-device state shared by every handle of the process
struct DeviceShared {
    std::mutex m;
    bool ready = false;
    int sm_count = 0, max_smem_optin = 0;
    PFN_cuTensorMapEncodeTiled_v12000 encode_tiled = nullptr;
    ColorTables h_tables;
    ColorTables* d_tables = nullptr;
};
static DeviceShared& device_shared(int device) {
    static DeviceShared table[64];
    return table[device & 63];
}

extern "C" int pcm_abi_version(void) { return PCM_ABI_VERSION; }
extern "C" const char* pcm_last_error(void) { return g_last_error.c_str(); }

extern "C" int pcm_create(int device, pcm_handle** out) {
    if (!out) return fail(PCM_E_INVALID, "pcm_create: out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(PCM_E_CUDA, "pcm_create: no CUDA device (%s); this library has no CPU path",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= count) return fail(PCM_E_INVALID, "pcm_create: device %d out of range [0,%d)", device, count);
    CUDA_TRY(cudaSetDevice(device));
    // once per device and process: device attributes, the driver entry point, the colour tables and the kernels'
    // shared-memory opt-in (a sweep creates one handle per sequence; none of this may cost per handle)
    DeviceShared& ds = device_shared(device);
    {
        std::lock_guard<std::mutex> lk(ds.m);
        if (!ds.ready) {
            CUDA_TRY(cudaDeviceGetAttribute(&ds.sm_count, cudaDevAttrMultiProcessorCount, device));
            CUDA_TRY(cudaDeviceGetAttribute(&ds.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
            void* fn = nullptr;
            cudaDriverEntryPointQueryResult qres;
            CUDA_TRY(cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &fn, 12000, cudaEnableDefault, &qres));
            if (qres != cudaDriverEntryPointSuccess || !fn)
                return fail(PCM_E_CUDA, "pcm_create: driver does not provide cuTensorMapEncodeTiled");
            ds.encode_tiled = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
            build_tables(ds.h_tables);
            CUDA_TRY(cudaMalloc(&ds.d_tables, sizeof(ColorTables)));
            CUDA_TRY(cudaMemcpy(ds.d_tables, &ds.h_tables, sizeof(ColorTables), cudaMemcpyHostToDevice));
            for (int i = 0; i < N_SCORE_VARIANTS; ++i)
                CUDA_TRY(cudaFuncSetAttribute(score_variant(i).fn, cudaFuncAttributeMaxDynamicSharedMemorySize, ds.max_smem_optin));
            CUDA_TRY(cudaFuncSetAttribute(qs_density_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ds.max_smem_optin));
            CUDA_TRY(cudaFuncSetAttribute(qs_density_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ds.max_smem_optin));
            CUDA_TRY(cudaFuncSetAttribute(qs_parent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ds.max_smem_optin));
            CUDA_TRY(cudaFuncSetAttribute(novelty_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ds.max_smem_optin));
            // once per device, never per call: the fits of a sweep run in several threads with different feature counts,
            // and a per-call limit set by one thread could undercut another thread's launch
            for (ResidualFn fn : pca_residual_kernels)
                CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, ds.max_smem_optin));
            ds.ready = true;
        }
    }
    pcm_handle* h = new pcm_handle();
    h->device = device;
    h->sm_count = ds.sm_count;
    h->max_smem_optin = ds.max_smem_optin;
    h->encode_tiled = ds.encode_tiled;
    h->d_tables = ds.d_tables;          // shared, never freed
    h->h_tables = ds.h_tables;
    CUDA_TRY(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    CUDA_TRY(h->err_buf.reserve(sizeof(int)));
    h->d_err = h->err_buf.as<int>();
    CUDA_TRY(cudaMemsetAsync(h->d_err, 0, sizeof(int), h->stream));
    *out = h;
    return PCM_OK;
}

// Named here, after the kernels of pcm_create: nvcc lays template kernels out in reverse order of first use, and this
// order keeps the SASS of the library (cuobjdump -sass) byte-identical to builds that named them inside pcm_create.
namespace {
const ResidualFn pca_residual_kernels[PCM_MAX_PCA_COMPONENTS] = {
    pca_residual_kernel<1>, pca_residual_kernel<2>, pca_residual_kernel<3>, pca_residual_kernel<4>,
    pca_residual_kernel<5>, pca_residual_kernel<6>, pca_residual_kernel<7>, pca_residual_kernel<8>};
}

extern "C" void pcm_destroy(pcm_handle* h) {
    if (!h) return;
    h->trace.report();
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    for (auto& t : h->pending) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
    for (cudaEvent_t e : h->band_events) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : h->feed_events) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ahead_events) if (e) cudaEventDestroy(e);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    for (auto e : h->free_events) cudaEventDestroy(e);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;                           // releases the models and every buffer, after the synchronisation above
}

extern "C" int pcm_set_stream(pcm_handle* h, void* cuda_stream) {
    if (!h) return fail(PCM_E_INVALID, "pcm_set_stream: NULL handle");
    h->stream = static_cast<cudaStream_t>(cuda_stream);
    h->chain_tail = false;
    return PCM_OK;
}

extern "C" int pcm_use_own_stream(pcm_handle* h) {
    if (!h) return fail(PCM_E_INVALID, "pcm_use_own_stream: NULL handle");
    h->stream = h->own_stream;
    h->chain_tail = false;
    return PCM_OK;
}

extern "C" int pcm_get_stream(const pcm_handle* h, void** out) {
    if (!h || !out) return fail(PCM_E_INVALID, "pcm_get_stream: NULL argument");
    *out = static_cast<void*>(h->stream);
    return PCM_OK;
}

// The error word is sticky on the device (no kernel clears it): an out-of-range label in ANY frame queued
// since the last check is reported here, then the word is cleared.
static int check_label_error(pcm_handle* h) {
    CUDA_TRY(h->h_small.reserve(64));      // the device-pointer entry points never touch the pinned scratch
    int* hs = h->h_small.as<int>();
    CUDA_TRY(cudaMemcpyAsync(hs, h->d_err, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    h->chain_tail = false;
    if (*hs) {
        CUDA_TRY(cudaMemsetAsync(h->d_err, 0, sizeof(int), h->stream));
        return fail(PCM_E_LABEL, "label outside [0, n_labels) in the label map");
    }
    return PCM_OK;
}

extern "C" int pcm_synchronize(pcm_handle* h) {
    if (!h) return fail(PCM_E_INVALID, "pcm_synchronize: NULL handle");
    CUDA_TRY(cudaSetDevice(h->device));
    return check_label_error(h);
}

// ---------------------------------------------------------------------------------
// API: configuration and models
// ---------------------------------------------------------------------------------
extern "C" int pcm_set_features(pcm_handle* h, int n_neighbors, int n_spaces, const int* space_ids) {
    if (!h || !space_ids) return fail(PCM_E_INVALID, "pcm_set_features: NULL argument");
    if (n_neighbors < 1 || n_neighbors > MAX_NEIGHBORS)
        return fail(PCM_E_LIMIT, "pcm_set_features: n_neighbors %d outside [1,%d]", n_neighbors, MAX_NEIGHBORS);
    if (n_spaces < 1 || n_spaces > MAX_SPACES)
        return fail(PCM_E_LIMIT, "pcm_set_features: n_spaces %d outside [1,%d]", n_spaces, MAX_SPACES);
    for (int i = 0; i < n_spaces; ++i)
        if (space_ids[i] < 0 || space_ids[i] > 2) return fail(PCM_E_INVALID, "pcm_set_features: bad space id %d", space_ids[i]);
    if (!h->models.empty()) return fail(PCM_E_STATE, "pcm_set_features: models already added (tap offsets are baked in)");
    h->geom = make_geom(n_neighbors, n_spaces, space_ids);
    h->features_set = true;
    return PCM_OK;
}

extern "C" int pcm_num_features(const pcm_handle* h) { return (h && h->features_set) ? h->geom.F : 0; }
extern "C" int pcm_num_models(const pcm_handle* h) { return h ? (int)h->models.size() : 0; }

extern "C" int pcm_add_model(pcm_handle* h, int n_frame, int n_trees, const int64_t* tree_offsets,
                             const int32_t* feature, const double* threshold, const int32_t* left,
                             const int32_t* right, const double* value1, int* model_index) {
    if (!h || !tree_offsets || !feature || !threshold || !left || !right || !value1)
        return fail(PCM_E_INVALID, "pcm_add_model: NULL argument");
    if (!h->features_set) return fail(PCM_E_STATE, "pcm_add_model: call pcm_set_features first");
    if (n_trees < 1) return fail(PCM_E_INVALID, "pcm_add_model: n_trees %d", n_trees);
    CUDA_TRY(cudaSetDevice(h->device));
    std::vector<NodeT> nodes;
    std::vector<double> leaves;
    std::vector<int4> trees;
    int max_depth = 0, n_leaf = 0;
    for (int t = 0; t < n_trees; ++t) {
        const int64_t b = tree_offsets[t], e = tree_offsets[t + 1];
        if (e <= b) return fail(PCM_E_INVALID, "pcm_add_model: tree %d is empty", t);
        Encoder enc{h->geom, feature + b, threshold + b, left + b, right + b, value1 + b, (int)(e - b)};
        if (!enc.run()) return fail(PCM_E_LIMIT, "pcm_add_model: tree %d: %s", t, enc.err.c_str());
        const unsigned base = (unsigned)nodes.size();       // entry index of this tree's root
        trees.push_back(make_int4((int)(NODE_BYTES * base), enc.out.depth, 0, 0));
        for (NodeT nd : enc.out.nodes) {
            node_set_left(nd, NODE_BYTES * (node_left(nd) + base));   // forest-relative byte offset
            nodes.push_back(nd);
        }
        leaves.insert(leaves.end(), enc.out.values.begin(), enc.out.values.end());
        max_depth = std::max(max_depth, enc.out.depth);
        n_leaf += enc.out.n_leaf;
    }
    if (nodes.size() > (1u << 26)) return fail(PCM_E_LIMIT, "pcm_add_model: forest too large");
    Model m;
    m.n_frame = n_frame;
    m.max_depth = max_depth;
    // one block, one copy: [nodes | leaves | trees], every part 16-byte aligned
    const size_t nb = (nodes.size() * sizeof(NodeT) + 15) / 16 * 16, lb = (leaves.size() * sizeof(double) + 15) / 16 * 16,
                 tb = trees.size() * sizeof(int4);
    std::vector<char> host(nb + lb + tb);
    memcpy(host.data(), nodes.data(), nodes.size() * sizeof(NodeT));
    memcpy(host.data() + nb, leaves.data(), leaves.size() * sizeof(double));
    memcpy(host.data() + nb + lb, trees.data(), tb);
    CUDA_TRY(m.blob.reserve(host.size()));
    CUDA_TRY(cudaMemcpyAsync(m.blob.p, host.data(), host.size(), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    m.forest.nodes = reinterpret_cast<const NodeT*>(m.blob.as<char>());
    m.forest.leaves = reinterpret_cast<const double*>(m.blob.as<char>() + nb);
    m.forest.trees = reinterpret_cast<const int4*>(m.blob.as<char>() + nb + lb);
    m.forest.n_trees = n_trees;
    m.forest.n_nodes = (int)nodes.size();
    m.forest.n_leaves = n_leaf;
    for (int t = 0; t < n_trees && t < MAX_TOP_TREES; ++t) {
        const NodeT root = nodes[trees[t].x / NODE_BYTES];
        const bool root_is_leaf = node_left(root) == (unsigned)trees[t].x;     // pseudo-node: left = self
        m.top.n[t][0] = root;
        m.top.n[t][1] = root_is_leaf ? root : nodes[node_left(root) / NODE_BYTES];
        m.top.n[t][2] = root_is_leaf ? root : nodes[node_left(root) / NODE_BYTES + 1];
    }
    h->models.push_back(std::move(m));      // the forest pointers into m.blob stay valid: the block moves, not its bytes
    if (model_index) *model_index = (int)h->models.size() - 1;
    return PCM_OK;
}

static_assert(MAX_PCA_K == PCM_MAX_PCA_COMPONENTS, "novelty_kernel and the C ABI disagree on the component limit");

extern "C" int pcm_set_novelty_k(pcm_handle* h, int model_index, const double* mean, const double* components,
                                 int n_components, int n_features) {
    if (!h || !mean || !components) return fail(PCM_E_INVALID, "pcm_set_novelty_k: NULL argument");
    if (n_components < 1) return fail(PCM_E_INVALID, "pcm_set_novelty_k: n_components %d < 1", n_components);
    if (n_components > PCM_MAX_PCA_COMPONENTS)
        return fail(PCM_E_LIMIT, "pcm_set_novelty_k: n_components %d > PCM_MAX_PCA_COMPONENTS (%d)", n_components,
                    PCM_MAX_PCA_COMPONENTS);
    if (model_index < 0 || model_index >= (int)h->models.size())
        return fail(PCM_E_INVALID, "pcm_set_novelty_k: model %d does not exist", model_index);
    if (n_features != h->geom.F) return fail(PCM_E_INVALID, "pcm_set_novelty_k: n_features %d != F %d", n_features, h->geom.F);
    CUDA_TRY(cudaSetDevice(h->device));
    Model& m = h->models[model_index];
    const Geom& g = h->geom;
    const int F = g.F, k = n_components, nch = 3 * g.n_spaces;
    // rank 1: K1's vectors in feature order
    if (k == 1) {
        std::vector<double> buf(3 * (size_t)F);
        double mdc = 0.0;
        for (int f = 0; f < F; ++f) {
            buf[f] = components[f];
            buf[F + f] = components[f] / 255.0;
            buf[2 * F + f] = mean[f];
            mdc += mean[f] * components[f];
        }
        CUDA_TRY(m.pca_buf.reserve(buf.size() * sizeof(double)));
        CUDA_TRY(cudaMemcpyAsync(m.pca_buf.p, buf.data(), buf.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        m.pca.comp = m.pca_buf.as<double>();
        m.pca.comp255 = m.pca.comp + F;
        m.pca.mean = m.pca.comp + 2 * F;
        m.pca.mean_dot_comp = mdc;
    } else {
        m.pca = DevPCA{};
    }
    // any rank: novelty_kernel's coefficients in its visiting order (a rank-1 model blended with a higher-rank one is
    // scored there too)
    std::vector<double> kb((size_t)F * (k + 1));
    for (int it = 0; it < F; ++it) {
        const int tap = it / nch, p = it - tap * nch;
        const int f = (p / 3) * 3 * g.K + 3 * tap + (p % 3);
        for (int j = 0; j < k; ++j) kb[(size_t)it * (k + 1) + j] = components[(size_t)j * F + f];
        kb[(size_t)it * (k + 1) + k] = mean[f];
    }
    for (int j = 0; j < MAX_PCA_K; ++j) {
        double mdc = 0.0;
        if (j < k)
            for (int f = 0; f < F; ++f) mdc += mean[f] * components[(size_t)j * F + f];
        m.pcak_mdc[j] = mdc;
    }
    CUDA_TRY(m.pcak_buf.reserve(kb.size() * sizeof(double)));
    CUDA_TRY(cudaMemcpyAsync(m.pcak_buf.p, kb.data(), kb.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    m.pca_k = k;
    m.has_pca = true;
    return PCM_OK;
}

extern "C" int pcm_set_novelty(pcm_handle* h, int model_index, const double* mean, const double* component,
                               int n_features) {
    if (!h || !mean || !component) return fail(PCM_E_INVALID, "pcm_set_novelty: NULL argument");
    return pcm_set_novelty_k(h, model_index, mean, component, 1, n_features);
}

// ---------------------------------------------------------------------------------
// API: per-frame hot path
// ---------------------------------------------------------------------------------
extern "C" int pcm_crop_rect(const int bbox[4], int H, int W, int rect_out[4]) {
    if (!bbox || !rect_out) return fail(PCM_E_INVALID, "pcm_crop_rect: NULL argument");
    const int e = 20;   // enlarge_bbox, pixel_classification.py:49
    const long long x = std::max(bbox[0] - e, 0), y = std::max(bbox[1] - e, 0);
    const long long w = std::min((long long)bbox[0] + bbox[2] + e, (long long)W) - bbox[0] + e;
    const long long hh = std::min((long long)bbox[1] + bbox[3] + e, (long long)H) - bbox[1] + e;
    // numpy slice a[start:start+len] with start >= 0: a negative stop counts from the end
    auto clamp = [](long long start, long long len, long long size, int& o0, int& o1) {
        long long stop = start + len;
        if (stop < 0) stop = std::max(size + stop, 0LL);
        o0 = (int)std::min(start, size);
        o1 = (int)std::min(std::max(stop, 0LL), size);
        if (o1 < o0) o1 = o0;
    };
    int x0, x1, y0, y1;
    clamp(x, w, W, x0, x1);
    clamp(y, hh, H, y0, y1);
    rect_out[0] = x0; rect_out[1] = y0; rect_out[2] = x1 - x0; rect_out[3] = y1 - y0;
    return PCM_OK;
}

static int check_rect(const char* who, const int rect[4], int H, int W) {
    if (rect[2] <= 0 || rect[3] <= 0 || rect[0] < 0 || rect[1] < 0 || rect[0] + rect[2] > W || rect[1] + rect[3] > H)
        return fail(PCM_E_INVALID, "%s: crop rect {%d,%d,%d,%d} is empty or outside the %dx%d frame", who, rect[0], rect[1],
                    rect[2], rect[3], W, H);
    return PCM_OK;
}

static int validate_update(pcm_handle* h, int H, int W, const int rect[4], int n_labels, const pcm_update_params* p) {
    if (!h->features_set) return fail(PCM_E_STATE, "update: call pcm_set_features first");
    if (!rect || !p) return fail(PCM_E_INVALID, "update: NULL argument");
    if (H <= 0 || W <= 0) return fail(PCM_E_INVALID, "update: bad frame size %dx%d", W, H);
    if (int rc = check_rect("update", rect, H, W)) return rc;
    if ((long long)rect[2] * rect[3] > (1LL << 30)) return fail(PCM_E_LIMIT, "update: crop too large");
    if (n_labels < 1) return fail(PCM_E_INVALID, "update: n_labels %d", n_labels);
    const int M = (int)h->models.size();
    if (p->model_cur < 0 || p->model_cur >= M) return fail(PCM_E_INVALID, "update: model_cur %d of %d", p->model_cur, M);
    if (p->model_next >= M || p->model_next < -1) return fail(PCM_E_INVALID, "update: model_next %d of %d", p->model_next, M);
    if (p->novelty) {
        if (!h->models[p->model_cur].has_pca) return fail(PCM_E_STATE, "update: novelty on but model %d has no PCA", p->model_cur);
        if (p->model_next >= 0 && !h->models[p->model_next].has_pca)
            return fail(PCM_E_STATE, "update: novelty on but model %d has no PCA", p->model_next);
    }
    if (p->dilation_kernel < 1 || p->dilation_kernel > DIL_MAXK)
        return fail(PCM_E_LIMIT, "update: dilation_kernel %d outside [1,%d]", p->dilation_kernel, DIL_MAXK);
    return PCM_OK;
}

// Enqueue K1..K3 for one crop.  All pointers are device pointers.
// rows of `width` bytes, `spitch` / `dpitch` apart: ONE flat copy when both sides are contiguous (a 2-D copy of a
// page-locked caller buffer runs row by row and was measured at about half the PCIe rate)
static cudaError_t copy_rows_async(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t height,
                                   cudaMemcpyKind kind, cudaStream_t st) {
    if (height == 0 || width == 0) return cudaSuccess;
    if (dpitch == width && spitch == width) return cudaMemcpyAsync(dst, src, width * height, kind, st);
    return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, height, kind, st);
}

// CTAs per SM of an NTHREADS-thread kernel at `smem` bytes of dynamic shared memory, queried once per (kernel, size): the
// runtime call costs more than launching a small crop's kernel
static cudaError_t occupancy(const void* kernel, size_t smem, int* occ) {
    static std::mutex m;
    static std::vector<std::pair<std::pair<const void*, size_t>, int>> cache;
    std::lock_guard<std::mutex> lk(m);
    const std::pair<const void*, size_t> key{kernel, smem};
    for (auto& e : cache)
        if (e.first == key) { *occ = e.second; return cudaSuccess; }
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, kernel, NTHREADS, smem);
    if (e != cudaSuccess) return e;
    *occ = std::max(*occ, 1);
    if (cache.size() < 4096) cache.push_back({key, *occ});
    return cudaSuccess;
}

// feed != NULL (host path with a page-locked caller frame): the crop rows are not on the device yet.  They are copied in a
// few row bands on the handle's copy stream, and the colour conversion (K0) and scoring (K1) of a band start as soon as its
// rows (plus the vertical halo of its last tile row) have arrived -- the copy of band b+1 overlaps the kernels of band b.
struct BandFeed {
    const uint8_t* src;       // first byte of the crop in the caller's frame
    size_t spitch;            // bytes between its rows
};
static int enqueue_update(pcm_handle* h, const uint8_t* d_frame, int H, int W, int64_t stride, const int rect[4],
                          const int32_t* d_labels, int S, const float* d_priors, const pcm_update_params* p,
                          uint8_t* d_mask, int64_t mask_stride, int mask_cx, int mask_cy, bool want_pre,
                          const BandFeed* feed = nullptr) {
    const int cx = rect[0], cy = rect[1], cw = rect[2], ch = rect[3];
    const size_t npx = (size_t)cw * ch;
    cudaStream_t st = h->stream;
    // the per-pixel P(fg) / novelty maps are kept only for pcm_debug_last (pcm_set_debug); K2 recomputes what it needs
    const bool keep_maps = want_pre;
    if (keep_maps) {
        CUDA_TRY(h->p1.reserve(npx * sizeof(double)));
        if (p->novelty) CUDA_TRY(h->sa.reserve(npx * sizeof(double)));
    }
    const SegLayout sl = seg_layout(S);
    CUDA_TRY(h->seg.reserve(sl.total));
    CUDA_TRY(h->rmin.reserve(sizeof(int) * (size_t)S));
    CUDA_TRY(h->rmax.reserve(sizeof(int) * (size_t)S));
    CUDA_TRY(h->cmin.reserve(sizeof(int) * (size_t)S));
    CUDA_TRY(h->cmax.reserve(sizeof(int) * (size_t)S));
    CUDA_TRY(h->decision.reserve((size_t)S));
    CUDA_TRY(h->scores.reserve(sizeof(float) * (size_t)S));
    if (want_pre) CUDA_TRY(h->pre.reserve(npx));

    // ---- K0: BGR crop -> planar colour planes (+ validity plane) ------------------------
    const Geom& g = h->geom;
    const long long pitch = ((long long)cw + 127) / 128 * 128;        // bytes
    const long long plane_stride = pitch * ch;                         // bytes
    CUDA_TRY(h->planes.reserve((size_t)plane_stride * g.n_planes));
    CUDA_TRY(h->sched.reserve(64));
    PlanesArgs pa{};
    pa.frame = d_frame;
    pa.stride = stride;
    pa.cx = cx; pa.cy = cy; pa.cw = cw; pa.ch = ch;
    pa.g = g;
    pa.tables = h->d_tables;
    pa.planes = h->planes.as<uint8_t>();
    pa.pitch = pitch;
    pa.plane_stride = plane_stride;
    pa.tile_counter = h->sched.as<unsigned>();
    char* seg = h->seg.as<char>();
    pa.n_labels = S;
    pa.sum = reinterpret_cast<double*>(seg + sl.sum);
    pa.asum = reinterpret_cast<double*>(seg + sl.asum);
    pa.area = reinterpret_cast<int*>(seg + sl.area);
    pa.rmin = h->rmin.as<int>();
    pa.rmax = h->rmax.as<int>();
    pa.cmin = h->cmin.as<int>();
    pa.cmax = h->cmax.as<int>();
    pa.n_flagged = reinterpret_cast<int*>(seg + sl.nflag);
    pa.early = (pdl_enabled() && st == h->own_stream && h->chain_tail && !feed) ? 1 : 0;
    // rows [r0, r1) of the crop; only the first launch of a frame resets the per-label accumulators
    auto launch_k0 = [&](int r0, int r1, bool first) -> int {
        PlanesArgs b = pa;
        b.cy = cy + r0;
        b.ch = r1 - r0;
        b.planes = pa.planes + (long long)r0 * pitch;
        if (!first) b.n_labels = 0;
        b.reset_flagged = first ? 1 : 0;
        // persistent blocks, 4 per SM: the 6.6 KB of lookup tables are staged once per block, so a block
        // should convert many pixel groups
        const long long groups = (long long)(r1 - r0) * ((cw + 3) / 4);
        const int blocks = (int)std::min<long long>((groups + 255) / 256, (long long)h->sm_count * 4);
        const int mode = (g.n_spaces == 2 && g.space_id[0] == PCM_SPACE_HSV && g.space_id[1] == PCM_SPACE_LAB) ? 1
                         : (g.n_spaces == 1 && g.space_id[0] == PCM_SPACE_LAB) ? 2 : 0;
        typedef void (*PlanesFn)(const PlanesArgs);
        static const PlanesFn table[3] = {planes_kernel<0>, planes_kernel<1>, planes_kernel<2>};
        return launch_timed(h, 6, "planes_kernel", table[mode], dim3(std::max(blocks, 1)), dim3(256), 0, b);
    };

    // ---- K1: TMA-tiled star features + forest(s) [+ novelty] -> P(fg) ------------------------
    ScoreArgs a{};
    a.cw = cw; a.ch = ch;
    a.tiles_x = (cw + TILE_W - 1) / TILE_W;
    a.g = g;
    a.tile_counter = h->sched.as<unsigned>();
    const Model& m0 = h->models[p->model_cur];
    a.f0 = m0.forest;
    a.top0 = m0.top;
    a.blend = p->model_next >= 0;
    a.depth = m0.max_depth;
    if (a.blend) {
        a.f1 = h->models[p->model_next].forest;
        a.top1 = h->models[p->model_next].top;
        a.depth = std::max(a.depth, h->models[p->model_next].max_depth);
    }
    a.w0 = p->w_cur; a.w1 = p->w_next;
    // a PCA of rank >= 2 on either model: novelty_kernel computes the (blended) error map between K0 and K1, which K1 and
    // K2 read; otherwise K1's in-line rank-1 pass
    const Model* m1 = a.blend ? &h->models[p->model_next] : nullptr;
    const bool nov_k = p->novelty != 0 && (m0.pca_k > 1 || (m1 && m1->pca_k > 1));
    a.novelty = p->novelty != 0;
    if (a.novelty && !nov_k) {
        a.pca0 = m0.pca;
        if (a.blend) a.pca1 = m1->pca;
    }
    NoveltyArgs na{};
    if (nov_k) {
        CUDA_TRY(h->sa.reserve(npx * sizeof(double)));
        a.nov_in = h->sa.as<double>();
        na.g = g;
        na.cw = cw; na.ch = ch;
        na.coef0 = m0.pcak_buf.as<double>(); na.k0 = m0.pca_k;
        for (int j = 0; j < MAX_PCA_K; ++j) na.mdc0[j] = m0.pcak_mdc[j];
        na.blend = a.blend;
        if (m1) {
            na.coef1 = m1->pcak_buf.as<double>(); na.k1 = m1->pca_k;
            for (int j = 0; j < MAX_PCA_K; ++j) na.mdc1[j] = m1->pcak_mdc[j];
        }
        na.w0 = a.w0; na.w1 = a.w1;
        na.staged = (int)novelty_smem_bytes(g, na.k0, na.k1, a.blend, true) <= h->max_smem_optin;
        na.out = h->sa.as<double>();
    }
    a.p1_out = keep_maps ? h->p1.as<double>() : nullptr;
    a.sa_out = (keep_maps && a.novelty && !nov_k) ? h->sa.as<double>() : nullptr;
    a.seg.labels = d_labels;
    a.seg.n_labels = S;
    a.seg.thr = p->outlier_threshold;
    a.seg.sum = pa.sum; a.seg.asum = pa.asum; a.seg.area = pa.area;
    a.seg.rmin = pa.rmin; a.seg.rmax = pa.rmax; a.seg.cmin = pa.cmin; a.seg.cmax = pa.cmax; a.seg.err = h->d_err;

    // forests live in shared memory whenever one CTA's tiles + forests fit, else they are read through L1
    ScoreSmem ls = score_smem_layout(a.g, a.f0, a.f1, a.blend, a.novelty && !nov_k, true);
    const bool forest_smem = (int)ls.total <= h->max_smem_optin;
    if (!forest_smem) ls = score_smem_layout(a.g, a.f0, a.f1, a.blend, a.novelty && !nov_k, false);
    if ((int)ls.total > h->max_smem_optin)
        return fail(PCM_E_LIMIT, "update: tile needs %u B of shared memory (> %d)", ls.total, h->max_smem_optin);
    // Tile height.  Measured on B200 (profiles/README.md, round 2): the kernel is throughput-bound on pipes the co-resident
    // CTAs of an SM share, so a partially filled last round of tiles does NOT cost a whole round (an SM with one CTA left
    // runs it nearly twice as fast) -- the time follows the fluid model  max(1, tiles / slots) * t_tile(ppt)  with
    // t_tile ~ 0.4 + 0.075 * ppt (per-tile and per-tree overheads do not shrink with the rows): at 1080p 32-row tiles win
    // (108.4 us vs 116.8 / 115.5 us for 28 / 24 rows), and shorter tiles pay only for crops with fewer tiles than CTA slots,
    // where every CTA has a single tile and a shorter tile simply ends sooner.  PCM_PPT forces a height.
    int ppt = MAX_PPT, occ = 0;
    {
        static const int forced = [] { const char* e = getenv("PCM_PPT"); return e ? atoi(e) : 0; }();
        CUDA_TRY(occupancy(reinterpret_cast<const void*>(pick_score_variant(forest_smem, a.depth, MAX_PPT).fn), ls.total, &occ));
        const double slots = (double)h->sm_count * occ;
        double best = -1.0;
        for (int c = MAX_PPT; c >= MIN_PPT; --c) {
            const double tiles = (double)a.tiles_x * ((ch + ROW_GROUPS * c - 1) / (ROW_GROUPS * c));
            const double cost = std::max(1.0, tiles / slots) * (0.4 + 0.075 * c);
            if (best < 0 || cost < best - 1e-9) { best = cost; ppt = c; }
        }
        if (forced >= MIN_PPT && forced <= MAX_PPT) ppt = forced;
    }
    const int tile_h = ROW_GROUPS * ppt;
    a.tiles_y = (ch + tile_h - 1) / tile_h;
    const ScoreVariant& sv = pick_score_variant(forest_smem, a.depth, ppt);
    CUDA_TRY(occupancy(reinterpret_cast<const void*>(sv.fn), ls.total, &occ));
    CUtensorMap tmap;
    {
        // planar u8 crop tensor {x, y, plane}; a box is ONE plane of a tile with its halo, zero fill outside the crop
        const cuuint64_t gdim[3] = {(cuuint64_t)cw, (cuuint64_t)ch, (cuuint64_t)g.n_planes};
        const cuuint64_t gstr[2] = {(cuuint64_t)pitch, (cuuint64_t)plane_stride};   // bytes
        const cuuint32_t box[3] = {(cuuint32_t)g.RS, (cuuint32_t)(tile_h + 2 * g.n), 1u};
        const cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = h->encode_tiled(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, h->planes.p, gdim, gstr, box, estr,
                                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(PCM_E_CUDA, "cuTensorMapEncodeTiled failed (%d) for a %dx%d crop", (int)r, cw, ch);
    }
    const int tiles_y = a.tiles_y;
    auto launch_k1 = [&](int ty0, int ty1) -> int {
        a.tile_y0 = ty0;
        a.tiles_y = ty1 - ty0;
        const int n_tiles = a.tiles_x * a.tiles_y;
        const int grid = std::min(n_tiles, h->sm_count * occ);
        return launch_timed(h, 0, sv.name, sv.fn, dim3(grid), dim3(NTHREADS), ls.total, tmap, a);
    };
    // novelty_kernel for the crop rows of K1's tile rows [ty0, ty1) (no launch unless a PCA of rank >= 2 is in use)
    auto launch_nk = [&](int ty0, int ty1) -> int {
        if (!nov_k) return PCM_OK;
        NoveltyArgs b = na;
        b.planes = pa.planes; b.pitch = pitch; b.plane_stride = plane_stride;
        b.row0 = ty0 * tile_h;
        b.rows = std::min(ch, ty1 * tile_h) - b.row0;
        const size_t smem = novelty_smem_bytes(g, b.k0, b.k1, b.blend != 0, b.staged != 0);
        int nk_occ = 0;
        CUDA_TRY(occupancy(reinterpret_cast<const void*>(novelty_kernel), smem, &nk_occ));
        const long long n_tiles = (long long)((cw + NOV_TW - 1) / NOV_TW) * ((b.rows + NOV_TH - 1) / NOV_TH);
        const int grid = (int)std::max<long long>(1, std::min<long long>(n_tiles, (long long)h->sm_count * nk_occ));
        return launch_timed(h, 7, "novelty_kernel", novelty_kernel, dim3(grid), dim3(NTHREADS), smem, b);
    };
    int rc = PCM_OK;
    if (!feed) {
        if ((rc = launch_k0(0, ch, true)) || (rc = launch_nk(0, tiles_y)) || (rc = launch_k1(0, tiles_y))) return rc;
    } else {
        // at most 2 bands of whole tile rows, at least ~512 Ki px each (measured at 1080p: 1 / 2 / 3 bands -> update
        // 0.434 / 0.429 / 0.471 ms); band b needs the crop rows up to the lower halo of its last tile row
        const int n_bands = (int)std::max<long long>(1, std::min<long long>({2LL, (long long)tiles_y, (long long)(npx >> 19)}));
        if (!h->copy_stream) CUDA_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        uint8_t* df = const_cast<uint8_t*>(d_frame);          // the handle's own crop buffer (rows `stride` apart)
        const size_t row_bytes = (size_t)cw * 3;
        int rows_done = 0;
        for (int b = 0; b < n_bands; ++b) {
            const int ty0 = (int)((long long)tiles_y * b / n_bands), ty1 = (int)((long long)tiles_y * (b + 1) / n_bands);
            const int rows_end = b + 1 == n_bands ? ch : std::min(ch, ty1 * tile_h + g.n);
            CUDA_TRY(copy_rows_async(df + (size_t)rows_done * stride, (size_t)stride, feed->src + (size_t)rows_done * feed->spitch, feed->spitch,
                                     row_bytes, (size_t)(rows_end - rows_done), cudaMemcpyHostToDevice, h->copy_stream));
            if (!h->feed_events[b]) CUDA_TRY(cudaEventCreateWithFlags(&h->feed_events[b], cudaEventDisableTiming));
            CUDA_TRY(cudaEventRecord(h->feed_events[b], h->copy_stream));
            CUDA_TRY(cudaStreamWaitEvent(st, h->feed_events[b], 0));
            if ((rc = launch_k0(rows_done, rows_end, b == 0)) || (rc = launch_nk(ty0, ty1)) || (rc = launch_k1(ty0, ty1))) return rc;
            rows_done = rows_end;
        }
        h->bytes_h2d += (int64_t)(npx * 3);
    }

    // ---- K2: per-label decision (+ exact path) ------------------------------------------------
    DecideArgs da{};
    da.p1 = a.p1_out; da.sa = nov_k && keep_maps ? a.nov_in : a.sa_out; da.labels = d_labels; da.cw = cw; da.thr = p->outlier_threshold;
    da.sum = pa.sum; da.asum = pa.asum; da.area = pa.area; da.rmin = pa.rmin; da.rmax = pa.rmax;
    da.cmin = pa.cmin; da.cmax = pa.cmax;
    da.ps.planes = pa.planes; da.ps.pitch = pitch; da.ps.plane_stride = plane_stride; da.ps.cw = cw; da.ps.ch = ch;
    da.ps.g = g; da.ps.f0 = a.f0; da.ps.f1 = a.f1; da.ps.depth = a.depth; da.ps.blend = a.blend;
    da.ps.w0 = a.w0; da.ps.w1 = a.w1; da.ps.novelty = a.novelty && !nov_k; da.ps.pca0 = a.pca0; da.ps.pca1 = a.pca1;
    da.ps.nov_map = a.nov_in;
    da.priors = d_priors;
    da.n_labels = S;
    da.prior_weight = p->prior_weight;
    da.decision = h->decision.as<uint8_t>();
    da.scores = h->scores.as<float>();
    da.n_flagged = reinterpret_cast<int*>(seg + sl.nflag);
    da.force_exact = h->force_exact ? 1 : 0;
    if ((rc = launch_timed(h, 2, "segment_decide_kernel", segment_decide_kernel, dim3((S + 255) / 256), dim3(256), 0, da))) return rc;

    // ---- K3 -------------------------------------------------------------------------
    DilateArgs dl{};
    dl.labels = d_labels;
    dl.decision = da.decision;
    dl.cw = cw; dl.ch = ch; dl.k = p->dilation_kernel; dl.n_labels = S;
    dl.mask = d_mask;
    dl.mask_stride = mask_stride;
    dl.cx = mask_cx; dl.cy = mask_cy;
    dl.pre = want_pre ? h->pre.as<uint8_t>() : nullptr;
    dim3 dg((cw + DIL_TW - 1) / DIL_TW, (ch + DIL_TH - 1) / DIL_TH);
    // 16-byte label loads need every label row to start on a 16-byte boundary
    const bool vec = (cw % 4 == 0) && (reinterpret_cast<uintptr_t>(d_labels) % 16 == 0);
    typedef void (*DilFn)(const DilateArgs);
    static const DilFn table[2][2][2] = {
        {{mask_dilate_kernel<false, false, 0>, mask_dilate_kernel<false, false, 7>},
         {mask_dilate_kernel<false, true, 0>, mask_dilate_kernel<false, true, 7>}},
        {{mask_dilate_kernel<true, false, 0>, mask_dilate_kernel<true, false, 7>},
         {mask_dilate_kernel<true, true, 0>, mask_dilate_kernel<true, true, 7>}}};
    if ((rc = launch_timed(h, 4, "mask_dilate_kernel", table[vec][dl.pre != nullptr][dl.k == 7], dg, dim3(256), 0, dl))) return rc;

    h->last_cw = cw; h->last_ch = ch; h->last_S = S;
    h->last_novelty = p->novelty != 0;      // rank 1: K1 wrote h->sa (maps kept); rank >= 2: novelty_kernel did
    h->last_valid = true;
    h->last_pre = want_pre;
    h->last_maps = keep_maps;
    h->chain_tail = true;
    return PCM_OK;
}

// (re)size the mask mirror for an H x W mask image; a new size forgets what was synchronised
static int ensure_mirror(pcm_handle* h, int H, int W) {
    if (h->mir_H == H && h->mir_W == W && h->mask.p && h->h_mask.p) return PCM_OK;
    const size_t n = (size_t)H * W;
    CUDA_TRY(h->h_mask.reserve(n));
    CUDA_TRY(h->mask.reserve(n));
    h->mir_H = H; h->mir_W = W;
    h->mir_band_rows = std::max(1, (int)((1u << 16) / (size_t)W));          // ~64 KiB bands: enough items to balance the pool
    h->mir_ok.assign((size_t)(H + h->mir_band_rows - 1) / h->mir_band_rows, 0);
    return PCM_OK;
}

// D2H of the crop region of the mask mirror in a few row bands; every band is scattered into the caller's (possibly
// interleaved) mask as soon as it has arrived, while the next one is still on the bus
static int finish_host_update(pcm_handle* h, const int rect[4], uint8_t* mask, int64_t mask_row_stride, int64_t mask_pixel_stride) {
    const int cx = rect[0], cy = rect[1], cw = rect[2], ch = rect[3], W = h->mir_W;
    const size_t npx = (size_t)cw * ch;
    cudaStream_t st = h->stream;
    uint8_t* hm = h->h_mask.as<uint8_t>();
    const uint8_t* dm = h->mask.as<uint8_t>();
    const int n_bands = (int)std::min<size_t>(4, std::max<size_t>(1, npx >> 19));    // >= 512 Ki px per band
    for (int b = 0; b < n_bands; ++b) {
        const int r0 = (int)((long long)ch * b / n_bands), r1 = (int)((long long)ch * (b + 1) / n_bands);
        const size_t o = (size_t)(cy + r0) * W + cx;
        CUDA_TRY(copy_rows_async(hm + o, (size_t)W, dm + o, (size_t)W, (size_t)cw, (size_t)(r1 - r0), cudaMemcpyDeviceToHost, st));
        if (b + 1 < n_bands) {
            if (!h->band_events[b]) CUDA_TRY(cudaEventCreateWithFlags(&h->band_events[b], cudaEventDisableTiming));
            CUDA_TRY(cudaEventRecord(h->band_events[b], st));
        }
    }
    h->bytes_d2h += (int64_t)npx + (int64_t)sizeof(int);
    HostPool& pool = HostPool::instance();
    for (int b = 0; b < n_bands; ++b) {
        if (b + 1 < n_bands) CUDA_TRY(cudaEventSynchronize(h->band_events[b]));
        else {
            int rc = check_label_error(h);                // last band: waits for the stream
            if (rc) return rc;
        }
        h->trace.lap(b == 0 ? HostTrace::UPD_WAIT : HostTrace::UPD_D2H);
        const int r0 = (int)((long long)ch * b / n_bands), r1 = (int)((long long)ch * (b + 1) / n_bands);
        const int parts = std::min(pool.size(), std::max(1, (int)(((size_t)(r1 - r0) * cw) >> 14)));
        pool.parallel_for(parts, [&](int part) {
            const int a0 = r0 + (int)((long long)(r1 - r0) * part / parts), a1 = r0 + (int)((long long)(r1 - r0) * (part + 1) / parts);
            for (int r = a0; r < a1; ++r)
                scatter_strided(hm + (size_t)(cy + r) * W + cx, mask + (size_t)(cy + r) * mask_row_stride + (size_t)cx * mask_pixel_stride,
                                mask_pixel_stride, cw);
        });
        h->trace.lap(HostTrace::UPD_SCATTER);
    }
    return PCM_OK;
}

// Rows [r0, r1) of a host image (row r at src + r * spitch, row_bytes each) packed densely into the pinned buffer `pin`,
// and their H2D copy into the same rows of the dense device buffer `dst` queued on the handle's stream
static cudaError_t stage_rows(pcm_handle* h, uint8_t* dst, uint8_t* pin, const uint8_t* src, size_t spitch, size_t row_bytes,
                              int r0, int r1) {
    for (int r = r0; r < r1; ++r) memcpy(pin + (size_t)r * row_bytes, src + (size_t)r * spitch, row_bytes);
    const size_t o = (size_t)r0 * row_bytes, n = (size_t)(r1 - r0) * row_bytes;
    const cudaError_t e = cudaMemcpyAsync(dst + o, pin + o, n, cudaMemcpyHostToDevice, h->stream);
    h->bytes_h2d += (int64_t)n;
    return e;
}

// rows of row_bytes each in a staging item of about chunk_bytes
static int rows_per_chunk(size_t chunk_bytes, size_t row_bytes) {
    return std::max(1, (int)(chunk_bytes / std::max<size_t>(row_bytes, 1)));
}

// One host-pool dispatch of n staging items on the handle's device: item(i) copies into pinned memory and returns the
// error of the H2D copy it queued.  Workers queue their copies themselves, so the DMA of finished items overlaps the
// staging of the others.
template <typename Item>
static int stage_items(pcm_handle* h, const char* who, int n, Item&& item) {
    std::atomic<int> cuda_err{0};
    const int device = h->device;
    HostPool::instance().parallel_for(n, [&](int i) {
        cudaSetDevice(device);
        const cudaError_t e = item(i);
        if (e != cudaSuccess) cuda_err.store((int)e);
    });
    if (cuda_err.load()) return fail(PCM_E_CUDA, "%s: staging copy failed: %s", who, cudaGetErrorString((cudaError_t)cuda_err.load()));
    return PCM_OK;
}

// n per-label priors -> pinned -> device.  The caller has synchronised the stream: the pinned buffer is reused between calls.
static int upload_priors(pcm_handle* h, const float* priors, int n, const float** d_priors) {
    const size_t bytes = sizeof(float) * (size_t)n;
    CUDA_TRY(h->h_priors.reserve(bytes));
    CUDA_TRY(h->priors.reserve(bytes));
    memcpy(h->h_priors.p, priors, bytes);
    CUDA_TRY(cudaMemcpyAsync(h->priors.p, h->h_priors.p, bytes, cudaMemcpyHostToDevice, h->stream));
    h->bytes_h2d += (int64_t)bytes;
    *d_priors = h->priors.as<float>();
    return PCM_OK;
}

// pcm_update(labels == NULL): the crop pixels and the label map are the ones the preceding
// pcm_quickshift or pcm_slic_gpu on this handle left on the device (h->handoff)
static int update_from_handoff(pcm_handle* h, const uint8_t* frame, int H, int W, int64_t stride, const int rect[4],
                               const float* priors, const pcm_update_params* params, uint8_t* mask,
                               int64_t mask_row_stride, int64_t mask_pixel_stride) {
    if (!rect) return fail(PCM_E_INVALID, "pcm_update: NULL rect");
    if (!h->handoff.valid || h->handoff.frame != frame || memcmp(h->handoff.rect, rect, sizeof h->handoff.rect) != 0)
        return fail(PCM_E_STATE, "pcm_update: labels == NULL needs a preceding pcm_quickshift or pcm_slic_gpu of the same frame and rect");
    int rc = validate_update(h, H, W, rect, h->handoff.n_labels, params);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(h->device));
    h->trace.start();
    const int cw = rect[2], ch = rect[3];
    rc = ensure_mirror(h, H, W);
    if (rc) return rc;
    CUDA_TRY(h->h_small.reserve(64));
    const float* d_priors = nullptr;
    if (priors) {
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        if ((rc = upload_priors(h, priors, h->handoff.n_labels, &d_priors))) return rc;
    }
    h->trace.lap(HostTrace::UPD_STAGE);
    const int crop_rect[4] = {0, 0, cw, ch};
    rc = enqueue_update(h, h->frame.as<uint8_t>(), ch, cw, (int64_t)cw * 3, crop_rect, h->seg_labels.as<int32_t>(),
                        h->handoff.n_labels, d_priors, params, h->mask.as<uint8_t>(), W, rect[0], rect[1], h->keep_pre);
    if (rc) return rc;
    h->trace.lap(HostTrace::UPD_ENQUEUE);
    return finish_host_update(h, rect, mask, mask_row_stride, mask_pixel_stride);
}

extern "C" int pcm_update_device(pcm_handle* h, const uint8_t* d_frame, int H, int W, int64_t stride, const int rect[4],
                                 const int32_t* d_labels, int n_labels, const float* d_priors,
                                 const pcm_update_params* params, uint8_t* d_mask, int64_t mask_row_stride) {
    if (!h || !d_frame || !d_labels || !d_mask) return fail(PCM_E_INVALID, "pcm_update_device: NULL argument");
    int rc = validate_update(h, H, W, rect, n_labels, params);
    if (rc) return rc;
    if (stride < (int64_t)W * 3) return fail(PCM_E_INVALID, "pcm_update_device: stride %lld < 3*W", (long long)stride);
    CUDA_TRY(cudaSetDevice(h->device));
    return enqueue_update(h, d_frame, H, W, stride, rect, d_labels, n_labels, d_priors, params, d_mask,
                          mask_row_stride, rect[0], rect[1], h->keep_pre);
}

extern "C" int pcm_update(pcm_handle* h, const uint8_t* frame, int H, int W, int64_t stride, const int rect[4],
                          const int32_t* labels, int n_labels, const float* priors, const pcm_update_params* params,
                          uint8_t* mask, int64_t mask_row_stride, int64_t mask_pixel_stride) {
    if (!h || !frame || !mask) return fail(PCM_E_INVALID, "pcm_update: NULL argument");
    if (!labels && h->handoff.valid) return update_from_handoff(h, frame, H, W, stride, rect, priors, params, mask, mask_row_stride, mask_pixel_stride);
    // labels == NULL without a pending handoff: the label map of the previous pcm_update (same crop size) is still on
    // the device and the caller vouches that it has not changed
    const bool reuse_labels = !labels;
    if (reuse_labels) {
        if (!rect || h->resident_labels <= 0 || rect[2] != h->resident_cw || rect[3] != h->resident_ch)
            return fail(PCM_E_STATE, "pcm_update: labels == NULL needs a preceding pcm_quickshift or pcm_slic_gpu of the same frame and rect, or a "
                                     "preceding pcm_update with a label map for a crop of the same size");
        n_labels = h->resident_labels;
    }
    h->handoff.valid = false;                          // the resident crop is about to be replaced
    h->chain_tail = false;
    const bool auto_labels = n_labels <= 0;            // n_labels = max(label) + 1, found while staging
    if (auto_labels && priors) return fail(PCM_E_INVALID, "pcm_update: priors need an explicit n_labels");
    int rc = validate_update(h, H, W, rect, auto_labels ? 1 : n_labels, params);
    if (rc) return rc;
    if (stride < (int64_t)W * 3) return fail(PCM_E_INVALID, "pcm_update: stride %lld < 3*W", (long long)stride);
    CUDA_TRY(cudaSetDevice(h->device));
    const int cx = rect[0], cy = rect[1], cw = rect[2], ch = rect[3];
    const size_t npx = (size_t)cw * ch, row_bytes = (size_t)cw * 3;
    cudaStream_t st = h->stream;
    h->trace.start();
    // host -> device: only the crop travels.  A crop inside a caller-registered (page-locked) range is copied
    // straight from the caller's memory, anything else goes through the handle's pinned staging buffer.
    const uint8_t* crop0 = frame + (size_t)cy * stride + (size_t)cx * 3;
    const bool direct = HostRegistry::instance().contains(crop0, (size_t)(ch - 1) * stride + row_bytes);
    const void* old_hl = h->h_labels.p;
    const void* old_dl = h->labels.p;
    if (!direct) CUDA_TRY(h->h_frame.reserve(npx * 3));
    CUDA_TRY(h->frame.reserve(npx * 3));
    if (!reuse_labels) CUDA_TRY(h->h_labels.reserve(npx * sizeof(int32_t)));
    CUDA_TRY(h->labels.reserve(npx * sizeof(int32_t)));
    rc = ensure_mirror(h, H, W);
    if (rc) return rc;
    CUDA_TRY(h->h_small.reserve(64));
    if (reuse_labels && old_dl != h->labels.p) return fail(PCM_E_STATE, "pcm_update: the resident label map was lost");
    CUDA_TRY(cudaStreamSynchronize(st));   // staging buffers are reused between calls
    h->trace.lap(HostTrace::UPD_SYNC);
    h->resident_labels = 0;

    uint8_t* df = h->frame.as<uint8_t>();
    const BandFeed feed{crop0, (size_t)stride};      // direct: enqueue_update copies the rows itself, band by band
    // One dispatch of the host pool stages everything else: an item is a ~1 MiB chunk of crop rows or
    // of the label map.  A label chunk whose bytes equal the previous call's (kept in the pinned buffer)
    // is neither copied nor re-sent.
    constexpr size_t CHUNK = 1u << 20;
    const int frame_rows = rows_per_chunk(CHUNK, row_bytes);
    const int n_frame_items = direct ? 0 : (ch + frame_rows - 1) / frame_rows;
    const size_t label_bytes = npx * sizeof(int32_t);
    const int n_label_items = reuse_labels ? 0 : (int)((label_bytes + CHUNK - 1) / CHUNK);
    const bool cache_ok = h->label_cache_on && h->label_cache_px == npx && old_hl == h->h_labels.p && old_dl == h->labels.p &&
                          (int)h->label_chunk_max.size() == n_label_items;
    if (!reuse_labels) {
        if (!cache_ok) h->label_chunk_max.assign(n_label_items, -1);
        h->label_cache_px = 0;                 // invalid until every chunk is staged
    }
    uint8_t* hf = h->h_frame.as<uint8_t>();
    uint8_t* hl = h->h_labels.as<uint8_t>();
    uint8_t* dl = h->labels.as<uint8_t>();
    const uint8_t* lsrc = reinterpret_cast<const uint8_t*>(labels);
    int* chunk_max = h->label_chunk_max.data();
    rc = stage_items(h, "pcm_update", n_frame_items + n_label_items, [&](int item) -> cudaError_t {
        if (item < n_frame_items) {
            const int r0 = item * frame_rows;
            return stage_rows(h, df, hf, crop0, (size_t)stride, row_bytes, r0, std::min(ch, r0 + frame_rows));
        }
        const int c = item - n_frame_items;
        const size_t o = (size_t)c * CHUNK, len = std::min(CHUNK, label_bytes - o);
        if (cache_ok && memcmp(hl + o, lsrc + o, len) == 0) return cudaSuccess;
        const int32_t* src = reinterpret_cast<const int32_t*>(lsrc + o);
        int32_t* dst = reinterpret_cast<int32_t*>(hl + o);
        int mx = -1;
        const size_t n = len / sizeof(int32_t);
        for (size_t i = 0; i < n; ++i) { const int32_t v = src[i]; dst[i] = v; mx = v > mx ? v : mx; }
        chunk_max[c] = mx;
        const cudaError_t e = cudaMemcpyAsync(dl + o, hl + o, len, cudaMemcpyHostToDevice, st);
        h->bytes_h2d += (int64_t)len;
        return e;
    });
    if (rc) return rc;
    if (!reuse_labels) {
        h->label_cache_px = npx;
        if (auto_labels) {
            int mx = -1;
            for (int c = 0; c < n_label_items; ++c) mx = std::max(mx, chunk_max[c]);
            if (mx < 0) return fail(PCM_E_LABEL, "pcm_update: label map has no non-negative label");
            n_labels = mx + 1;
        }
    }
    h->trace.lap(HostTrace::UPD_STAGE);
    const float* d_priors = nullptr;
    if (priors && (rc = upload_priors(h, priors, n_labels, &d_priors))) return rc;
    const int crop_rect[4] = {0, 0, cw, ch};
    rc = enqueue_update(h, h->frame.as<uint8_t>(), ch, cw, (int64_t)row_bytes, crop_rect, h->labels.as<int32_t>(),
                        n_labels, d_priors, params, h->mask.as<uint8_t>(), W, cx, cy, h->keep_pre, direct ? &feed : nullptr);
    if (rc) return rc;
    h->trace.lap(HostTrace::UPD_ENQUEUE);
    rc = finish_host_update(h, rect, mask, mask_row_stride, mask_pixel_stride);
    if (rc) return rc;
    h->resident_labels = n_labels;
    h->resident_cw = cw; h->resident_ch = ch;
    return PCM_OK;
}

static int enqueue_iou(pcm_handle* h, const uint8_t* d_mask, int64_t mask_row_stride, const uint8_t* d_truth,
                       int64_t truth_row_stride, int truth_channels, int height, int width, int64_t* d_counts, const int* valid);

extern "C" int pcm_iou_device(pcm_handle* h, const uint8_t* d_mask, int64_t mask_row_stride, const uint8_t* d_truth,
                              int64_t truth_row_stride, int truth_channels, int height, int width, int64_t* d_counts) {
    return enqueue_iou(h, d_mask, mask_row_stride, d_truth, truth_row_stride, truth_channels, height, width, d_counts, nullptr);
}

// valid: {x, y, w, h} rectangle outside of which the mask plane reads as zero, or NULL
static int enqueue_iou(pcm_handle* h, const uint8_t* d_mask, int64_t mask_row_stride, const uint8_t* d_truth,
                       int64_t truth_row_stride, int truth_channels, int height, int width, int64_t* d_counts, const int* valid) {
    if (!h || !d_mask || !d_truth || !d_counts) return fail(PCM_E_INVALID, "pcm_iou_device: NULL argument");
    if (truth_channels != 1 && truth_channels != 3) return fail(PCM_E_INVALID, "pcm_iou_device: truth_channels %d", truth_channels);
    if (height <= 0 || width <= 0) return fail(PCM_E_INVALID, "pcm_iou_device: bad size");
    CUDA_TRY(cudaSetDevice(h->device));
    const long long work = ((long long)height * width + 15) / 16;
    const int blocks = (int)std::min<long long>((work + 255) / 256, (long long)h->sm_count * 8);
    const int4 vr = valid ? make_int4(valid[0], valid[1], valid[2], valid[3]) : make_int4(0, 0, -1, -1);
    return launch_timed(h, 5, "iou_kernel", iou_kernel, dim3(std::max(blocks, 1)), dim3(256), 0, d_mask, (long long)mask_row_stride,
                        d_truth, (long long)truth_row_stride, truth_channels, height, width, vr,
                        reinterpret_cast<unsigned long long*>(d_counts));
}

extern "C" int pcm_iou(pcm_handle* h, const uint8_t* mask, int64_t mask_row_stride, int64_t mask_pixel_stride,
                       const uint8_t* truth, int64_t truth_row_stride, int truth_channels, int height, int width,
                       int64_t counts[2]) {
    if (!h || !mask || !truth || !counts) return fail(PCM_E_INVALID, "pcm_iou: NULL argument");
    if (truth_channels != 1 && truth_channels != 3) return fail(PCM_E_INVALID, "pcm_iou: truth_channels %d", truth_channels);
    if (height <= 0 || width <= 0) return fail(PCM_E_INVALID, "pcm_iou: bad size");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const size_t npx = (size_t)height * width, tbytes = npx * truth_channels;
    const size_t trow = (size_t)width * truth_channels;
    const bool direct = HostRegistry::instance().contains(truth, (size_t)(height - 1) * truth_row_stride + trow);
    int rc = ensure_mirror(h, height, width);
    if (rc) return rc;
    if (!direct) CUDA_TRY(h->h_frame.reserve(tbytes));
    CUDA_TRY(h->frame.reserve(tbytes));
    CUDA_TRY(h->counts.reserve(2 * sizeof(int64_t)));
    CUDA_TRY(h->h_small.reserve(64));
    CUDA_TRY(cudaStreamSynchronize(st));
    h->handoff.valid = false;                          // the frame scratch is reused for the truth image
    h->chain_tail = false;
    h->trace.start();
    uint8_t* hm = h->h_mask.as<uint8_t>();
    uint8_t* ht = h->h_frame.as<uint8_t>();
    uint8_t* dm = h->mask.as<uint8_t>();
    uint8_t* dt = h->frame.as<uint8_t>();
    if (direct) {
        CUDA_TRY(copy_rows_async(dt, trow, truth, (size_t)truth_row_stride, trow, (size_t)height, cudaMemcpyHostToDevice, st));
        h->bytes_h2d += (int64_t)tbytes;
    }
    // one pool dispatch: an item is a band of rows of the truth (packed densely into pinned memory, its H2D copy queued by
    // the worker) or of the mask.  A mask band is first COMPARED with the pinned mirror of what the device already holds
    // (the crop pcm_update produced, bands uploaded by an earlier call): only a band that differs is copied and re-sent.
    const int rows_t = rows_per_chunk(1u << 18, trow);      // 256 KiB bands: enough items for
    const int rows_m = h->mir_band_rows;                    // every pool thread at 1080p
    const int n_t = direct ? 0 : (height + rows_t - 1) / rows_t, n_m = (height + rows_m - 1) / rows_m;
    uint8_t* band_ok = h->mir_ok.data();
    std::atomic<int> refreshed{0};
    int64_t* hc = h->h_small.as<int64_t>() + 2;
    auto count = [&]() -> int {
        CUDA_TRY(cudaMemsetAsync(h->counts.p, 0, 2 * sizeof(int64_t), st));
        int r = pcm_iou_device(h, h->mask.as<uint8_t>(), width, h->frame.as<uint8_t>(), (int64_t)width * truth_channels,
                               truth_channels, height, width, h->counts.as<int64_t>());
        if (r) return r;
        CUDA_TRY(cudaMemcpyAsync(hc, h->counts.p, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        h->bytes_d2h += 2 * (int64_t)sizeof(int64_t);
        return PCM_OK;
    };
    // The truth is already on its way and every band of the mirror is believed to be current (the usual case right after
    // pcm_update): count NOW, on what the device holds, while the host threads verify the caller's bytes against the
    // mirror; only if a band turns out to differ is it re-sent and the count repeated.
    bool speculative = direct;
    for (int b = 0; b < n_m && speculative; ++b) speculative = band_ok[b] != 0;
    if (speculative) { rc = count(); if (rc) return rc; }
    rc = stage_items(h, "pcm_iou", n_t + n_m, [&](int item) -> cudaError_t {
        if (item < n_t) {
            const int r0 = item * rows_t;
            return stage_rows(h, dt, ht, truth, (size_t)truth_row_stride, trow, r0, std::min(height, r0 + rows_t));
        }
        const int b = item - n_t;
        const int r0 = b * rows_m, r1 = std::min(height, r0 + rows_m);
        int r = r0;
        if (band_ok[b]) {
            uint8_t tmp[4096];
            for (; r < r1; ++r) {                           // rows equal to the mirror need nothing
                const uint8_t* src = mask + (size_t)r * mask_row_stride;
                const uint8_t* have = hm + (size_t)r * width;
                bool same = true;
                if (mask_pixel_stride == 1) same = memcmp(src, have, (size_t)width) == 0;
                else
                    for (int c0 = 0; c0 < width && same; c0 += (int)sizeof tmp) {
                        const int n = std::min<int>((int)sizeof tmp, width - c0);
                        gather_strided(src + (size_t)c0 * mask_pixel_stride, mask_pixel_stride, tmp, n);
                        same = memcmp(tmp, have + c0, (size_t)n) == 0;
                    }
                if (!same) break;
            }
        }
        if (r == r1) return cudaSuccess;
        // from the first differing row on: refresh mirror and device
        for (int q = r; q < r1; ++q) gather_strided(mask + (size_t)q * mask_row_stride, mask_pixel_stride, hm + (size_t)q * width, width);
        const cudaError_t e = cudaMemcpyAsync(dm + (size_t)r * width, hm + (size_t)r * width, (size_t)(r1 - r) * width, cudaMemcpyHostToDevice, st);
        h->bytes_h2d += (int64_t)((size_t)(r1 - r) * width);
        band_ok[b] = 1;
        refreshed.store(1);
        return e;
    });
    if (rc) {
        h->mir_ok.assign(h->mir_ok.size(), 0);
        return rc;
    }
    h->trace.lap(HostTrace::IOU_STAGE);
    if (!speculative || refreshed.load()) { rc = count(); if (rc) return rc; }
    CUDA_TRY(cudaStreamSynchronize(st));
    h->trace.lap(HostTrace::IOU_WAIT);
    counts[0] = hc[0];
    counts[1] = hc[1];
    h->last_valid = false;   // frame scratch was reused
    return PCM_OK;
}

extern "C" int pcm_host_register(void* p, size_t bytes) {
    if (!p || !bytes) return fail(PCM_E_INVALID, "pcm_host_register: NULL / empty range");
    if (HostRegistry::instance().contains(p, bytes)) return PCM_OK;
    cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(PCM_E_CUDA, "pcm_host_register: cudaHostRegister failed: %s", cudaGetErrorString(e));
    }
    HostRegistry::instance().add(p, bytes);
    return PCM_OK;
}

extern "C" int pcm_host_unregister(void* p) {
    if (!p) return fail(PCM_E_INVALID, "pcm_host_unregister: NULL");
    if (!HostRegistry::instance().remove(p)) return fail(PCM_E_STATE, "pcm_host_unregister: %p was not registered here", p);
    CUDA_TRY(cudaHostUnregister(p));
    return PCM_OK;
}

// ---------------------------------------------------------------------------------
// over-segmentation on the GPU: the front end quickshift and SLIC share.  Each algorithm's enqueue_* queues it on a crop
// of a device frame, writes the label map into h->seg_labels and leaves its count in a device word.
// ---------------------------------------------------------------------------------
// The checks and set-up every entry point below starts with.  The handoff ends here: the call replaces the label map,
// and a host entry point also the staged crop.
static int begin_seg(pcm_handle* h, const char* who, const uint8_t* frame, int H, int W, int64_t stride, const int rect[4]) {
    if (!h || !frame || !rect) return fail(PCM_E_INVALID, "%s: NULL argument", who);
    if (int rc = check_rect(who, rect, H, W)) return rc;
    if (stride < (int64_t)W * 3) return fail(PCM_E_INVALID, "%s: stride %lld < 3*W", who, (long long)stride);
    CUDA_TRY(cudaSetDevice(h->device));
    h->handoff.valid = false;
    return PCM_OK;
}

// Waits for the stream; *n = the device word d_count + bias (0: quickshift counts its segments; 1: SLIC leaves its largest
// label, and pcm_slic counts largest label + 1)
static int read_seg_count(pcm_handle* h, const int* d_count, int bias, int* n) {
    CUDA_TRY(h->h_small.reserve(64));
    int* hs = h->h_small.as<int>() + 8;
    CUDA_TRY(cudaMemcpyAsync(hs, d_count, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    *n = *hs + bias;
    return PCM_OK;
}

// Host entry points, before the algorithm: the crop rows of the host frame -> pinned -> h->frame (dense rows of 3 * w
// bytes, where pcm_update with labels == NULL finds them), and n_extra items of the caller's in the same pool dispatch
// (extra(i) stages item i and returns the error of the copy it queued)
template <typename Extra>
static int stage_crop(pcm_handle* h, const char* who, const uint8_t* frame, int64_t stride, const int rect[4], int n_extra,
                      Extra&& extra) {
    const int ch = rect[3];
    const size_t row_bytes = (size_t)rect[2] * 3;
    CUDA_TRY(h->h_frame.reserve(row_bytes * ch));
    CUDA_TRY(h->frame.reserve(row_bytes * ch));
    CUDA_TRY(cudaStreamSynchronize(h->stream));       // the staging buffers are reused between calls
    const int frame_rows = rows_per_chunk((size_t)1 << 20, row_bytes);
    const int n_frame_items = (ch + frame_rows - 1) / frame_rows;
    const uint8_t* crop0 = frame + (size_t)rect[1] * stride + (size_t)rect[0] * 3;
    uint8_t* hf = h->h_frame.as<uint8_t>();
    uint8_t* df = h->frame.as<uint8_t>();
    return stage_items(h, who, n_frame_items + n_extra, [&](int item) -> cudaError_t {
        if (item >= n_frame_items) return extra(item - n_frame_items);
        const int r0 = item * frame_rows;
        return stage_rows(h, df, hf, crop0, (size_t)stride, row_bytes, r0, std::min(ch, r0 + frame_rows));
    });
}

// Host entry points, after the algorithm: the label map to labels_out (when given), the count (read_seg_count), and the
// handoff armed for this frame and rect
static int finish_host_seg(pcm_handle* h, const uint8_t* frame, const int rect[4], const int* d_count, int bias,
                           int32_t* labels_out, int* n_labels_out) {
    const size_t label_bytes = (size_t)rect[2] * rect[3] * sizeof(int32_t);
    if (labels_out) {
        CUDA_TRY(h->h_labels.reserve(label_bytes));
        h->label_cache_px = 0;                        // the pinned label buffer no longer mirrors `labels`
        CUDA_TRY(cudaMemcpyAsync(h->h_labels.p, h->seg_labels.p, label_bytes, cudaMemcpyDeviceToHost, h->stream));
        h->bytes_d2h += (int64_t)label_bytes;
    }
    int n = 0;
    if (int rc = read_seg_count(h, d_count, bias, &n)) return rc;
    if (n_labels_out) *n_labels_out = n;
    if (labels_out) memcpy(labels_out, h->h_labels.p, label_bytes);
    h->handoff = {true, frame, {rect[0], rect[1], rect[2], rect[3]}, n};
    return PCM_OK;
}

// Device entry points: enqueue() queues the algorithm on the crop `rect` of d_frame; the map is then copied into
// d_labels_out (when given) and the count read from h->*count (read_seg_count)
template <typename Enqueue>
static int seg_device(pcm_handle* h, const char* who, const uint8_t* d_frame, int H, int W, int64_t stride, const int rect[4],
                      DevBuf pcm_handle::*count, int bias, int32_t* d_labels_out, int* n_labels_out, Enqueue&& enqueue) {
    if (int rc = begin_seg(h, who, d_frame, H, W, stride, rect)) return rc;
    if (int rc = enqueue()) return rc;
    if (d_labels_out)
        CUDA_TRY(cudaMemcpyAsync(d_labels_out, h->seg_labels.p, (size_t)rect[2] * rect[3] * sizeof(int32_t), cudaMemcpyDeviceToDevice,
                                 h->stream));
    int n = 0;
    if (int rc = read_seg_count(h, (h->*count).as<int>(), bias, &n)) return rc;
    if (n_labels_out) *n_labels_out = n;
    return PCM_OK;
}

// The *_device_batch entry points: crop k = rects[4k .. 4k+3] of the frame d_frames + frame_index[k] * frame_bytes through
// one(d_frame, rect, d_labels, &count), the single-crop entry point, into d_labels_out + label_offsets[k]
template <typename One>
static int seg_device_batch(pcm_handle* h, const char* who, int n, const uint8_t* d_frames, int64_t frame_bytes,
                            const int32_t* frame_index, const int32_t* rects, int32_t* d_labels_out, const int64_t* label_offsets,
                            int32_t* n_labels_out, One&& one) {
    if (!h || !d_frames || !frame_index || !rects || !d_labels_out || !label_offsets || !n_labels_out)
        return fail(PCM_E_INVALID, "%s: NULL argument", who);
    if (n < 0 || frame_bytes < 0) return fail(PCM_E_INVALID, "%s: bad count / frame size", who);
    for (int k = 0; k < n; ++k) {
        if (frame_index[k] < 0 || label_offsets[k] < 0) return fail(PCM_E_INVALID, "%s: crop %d: negative index", who, k);
        int count = 0;
        const int rect[4] = {rects[4 * k], rects[4 * k + 1], rects[4 * k + 2], rects[4 * k + 3]};
        if (int rc = one(d_frames + (int64_t)frame_index[k] * frame_bytes, rect, d_labels_out + label_offsets[k], &count)) return rc;
        n_labels_out[k] = count;
    }
    return PCM_OK;
}

// ---------------------------------------------------------------------------------
// API: quickshift over-segmentation (SURVEY.md §8 f-1)
// ---------------------------------------------------------------------------------
static int enqueue_quickshift(pcm_handle* h, const uint8_t* d_frame, int64_t stride, int cx, int cy, int cw, int ch,
                              double ratio, double kernel_size, double max_dist, const double* d_noise) {
    if (!(kernel_size >= 1.0)) return fail(PCM_E_INVALID, "quickshift: kernel_size must be >= 1");
    const int kw = (int)ceil(3.0 * kernel_size);
    if (kw > QS_MAX_KW) return fail(PCM_E_LIMIT, "quickshift: window half width %d > %d", kw, QS_MAX_KW);
    const size_t n = (size_t)cw * ch;
    if (n > (1u << 30)) return fail(PCM_E_LIMIT, "quickshift: crop too large");
    cudaStream_t st = h->stream;
    h->chain_tail = false;
    CUDA_TRY(h->qs_lab.reserve(3 * n * sizeof(double)));
    CUDA_TRY(h->qs_dens.reserve(n * sizeof(double)));
    CUDA_TRY(h->qs_parent.reserve(n * sizeof(int)));
    CUDA_TRY(h->qs_root.reserve(n * sizeof(int)));
    CUDA_TRY(h->qs_flag.reserve(n * sizeof(int)));
    CUDA_TRY(h->qs_rank.reserve(n * sizeof(int)));
    const int n_blocks = (int)((n + QS_SCAN_ELEMS - 1) / QS_SCAN_ELEMS);
    CUDA_TRY(h->qs_sums.reserve((size_t)n_blocks * sizeof(int)));
    CUDA_TRY(h->seg_labels.reserve(n * sizeof(int32_t)));
    CUDA_TRY(h->qs_count.reserve(sizeof(int)));
    if (!h->qs_lin.p) {
        // sRGB companding table of skimage.color.rgb2xyz for the 256 byte values
        double lin[256];
        for (int v = 0; v < 256; ++v) {
            const double x = v / 255.0;
            lin[v] = x > 0.04045 ? pow((x + 0.055) / 1.055, 2.4) : x / 12.92;
        }
        // + the table of qs_exp_neg: 2^(j/64) as float64 high part and the remainder
        double tab[128];
        for (int j = 0; j < 64; ++j) {
            const long double v = exp2l((long double)j / 64.0L);
            tab[2 * j] = (double)v;
            tab[2 * j + 1] = (double)(v - (long double)tab[2 * j]);
        }
        CUDA_TRY(h->qs_lin.reserve(sizeof lin + sizeof tab));
        CUDA_TRY(cudaMemcpy(h->qs_lin.p, lin, sizeof lin, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(h->qs_lin.as<char>() + sizeof lin, tab, sizeof tab, cudaMemcpyHostToDevice));
    }
    QsArgs a{};
    a.frame = d_frame; a.stride = stride; a.cx = cx; a.cy = cy; a.cw = cw; a.ch = ch;
    a.lin = h->qs_lin.as<double>();
    a.ratio = ratio;
    a.lab = h->qs_lab.as<double>();
    a.dens = h->qs_dens.as<double>();
    a.noise = d_noise;
    a.parent = h->qs_parent.as<int>();
    a.root = h->qs_root.as<int>();
    a.kw = kw;
    a.inv = -0.5 / (kernel_size * kernel_size);
    a.max_dist = max_dist;
    a.exp_tab = h->qs_lin.as<double>() + 256;
    {
        // largest possible squared 5-D distance: Lab * ratio spans L 0..100, a / b about -128..128 (generous), plus the
        // window corner; the exp argument is that times |inv|
        const double span = ratio * ratio * (100.0 * 100.0 + 2.0 * 256.0 * 256.0) + 2.0 * (double)kw * kw;
        a.exp_guard = !(span * -a.inv < 690.0);
    }
    a.pw = (max_dist >= 0 && max_dist < (double)kw) ? (int)floor(max_dist) : kw;
    const int flat_blocks = (int)std::min<size_t>((n + 255) / 256, (size_t)h->sm_count * 16);
    qs_lab_kernel<<<flat_blocks, 256, 0, st>>>(a);
    CHECK_LAUNCH(h, "qs_lab_kernel");
    const dim3 grid((cw + QS_BW - 1) / QS_BW, (ch + QS_BH - 1) / QS_BH);
    {
        const dim3 dgrid((cw + QS_DBW - 1) / QS_DBW, (ch + QS_DBH - 1) / QS_DBH);
        const size_t dtile = (size_t)(QS_DBW + 2 * kw) * (QS_DBH + 2 * kw) * sizeof(double);
        const size_t dsmem = 3 * dtile + (128 + 2 * kw + 1) * sizeof(double);
        if (a.exp_guard) qs_density_kernel<true><<<dgrid, 256, dsmem, st>>>(a);
        else qs_density_kernel<false><<<dgrid, 256, dsmem, st>>>(a);
    }
    CHECK_LAUNCH(h, "qs_density_kernel");
    const size_t ptile = (size_t)(QS_BW + 2 * a.pw) * (QS_BH + 2 * a.pw) * sizeof(double);
    qs_parent_kernel<<<grid, QS_BW * QS_BH, 4 * ptile, st>>>(a);
    CHECK_LAUNCH(h, "qs_parent_kernel");
    CUDA_TRY(cudaMemsetAsync(h->qs_flag.p, 0, n * sizeof(int), st));
    qs_root_kernel<<<flat_blocks, 256, 0, st>>>(a.parent, a.root, h->qs_flag.as<int>(), (int)n);
    CHECK_LAUNCH(h, "qs_root_kernel");
    qs_scan_reduce_kernel<<<n_blocks, 256, 0, st>>>(h->qs_flag.as<int>(), (int)n, h->qs_sums.as<int>());
    CHECK_LAUNCH(h, "qs_scan_reduce_kernel");
    qs_scan_sums_kernel<<<1, 256, 0, st>>>(h->qs_sums.as<int>(), n_blocks, h->qs_count.as<int>());
    CHECK_LAUNCH(h, "qs_scan_sums_kernel");
    qs_scan_apply_kernel<<<n_blocks, 256, 0, st>>>(h->qs_flag.as<int>(), (int)n, h->qs_sums.as<int>(), h->qs_rank.as<int>());
    CHECK_LAUNCH(h, "qs_scan_apply_kernel");
    qs_label_kernel<<<flat_blocks, 256, 0, st>>>(a.root, h->qs_rank.as<int>(), h->seg_labels.as<int32_t>(), (int)n);
    CHECK_LAUNCH(h, "qs_label_kernel");
    return PCM_OK;
}

extern "C" int pcm_quickshift_device(pcm_handle* h, const uint8_t* d_frame, int H, int W, int64_t stride, const int rect[4],
                                     double ratio, double kernel_size, double max_dist, const double* d_noise,
                                     int32_t* d_labels_out, int* n_labels_out) {
    return seg_device(h, "pcm_quickshift_device", d_frame, H, W, stride, rect, &pcm_handle::qs_count, 0, d_labels_out, n_labels_out,
                      [&] {
                          return enqueue_quickshift(h, d_frame, stride, rect[0], rect[1], rect[2], rect[3], ratio, kernel_size,
                                                    max_dist, d_noise);
                      });
}

extern "C" int pcm_quickshift_device_batch(pcm_handle* h, int n, const uint8_t* d_frames, int64_t frame_bytes,
                                           const int32_t* frame_index, int H, int W, int64_t stride, const int32_t* rects,
                                           double ratio, double kernel_size, double max_dist, const double* d_noise,
                                           int32_t* d_labels_out, const int64_t* label_offsets, int32_t* n_labels_out) {
    return seg_device_batch(h, "pcm_quickshift_device_batch", n, d_frames, frame_bytes, frame_index, rects, d_labels_out, label_offsets,
                            n_labels_out, [&](const uint8_t* d_frame, const int rect[4], int32_t* d_labels, int* count) {
                                return pcm_quickshift_device(h, d_frame, H, W, stride, rect, ratio, kernel_size, max_dist, d_noise,
                                                             d_labels, count);
                            });
}

extern "C" int pcm_quickshift(pcm_handle* h, const uint8_t* frame, int H, int W, int64_t stride, const int rect[4],
                              double ratio, double kernel_size, double max_dist, const double* noise,
                              int32_t* labels_out, int* n_labels_out) {
    int rc = begin_seg(h, "pcm_quickshift", frame, H, W, stride, rect);
    if (rc) return rc;
    const int cw = rect[2], ch = rect[3];
    const size_t npx = (size_t)cw * ch;
    if (noise) {
        CUDA_TRY(h->h_noise.reserve(npx * sizeof(double)));
        CUDA_TRY(h->qs_noise.reserve(npx * sizeof(double)));
    } else if (h->qs_noise_cw != cw || h->qs_noise_ch != ch) {
        return fail(PCM_E_STATE, "pcm_quickshift: noise == NULL needs a previous call with noise for the same %dx%d crop", cw, ch);
    }
    // the tie-breaking noise, when given, travels with the crop rows
    constexpr size_t CHUNK = 1u << 20;
    const size_t noise_bytes = noise ? npx * sizeof(double) : 0;
    uint8_t* hn = h->h_noise.as<uint8_t>();
    uint8_t* dn = h->qs_noise.as<uint8_t>();
    const uint8_t* nsrc = reinterpret_cast<const uint8_t*>(noise);
    rc = stage_crop(h, "pcm_quickshift", frame, stride, rect, (int)((noise_bytes + CHUNK - 1) / CHUNK), [&](int item) -> cudaError_t {
        const size_t o = (size_t)item * CHUNK, len = std::min(CHUNK, noise_bytes - o);
        memcpy(hn + o, nsrc + o, len);
        const cudaError_t e = cudaMemcpyAsync(dn + o, hn + o, len, cudaMemcpyHostToDevice, h->stream);
        h->bytes_h2d += (int64_t)len;
        return e;
    });
    if (rc) return rc;
    if (noise) { h->qs_noise_cw = cw; h->qs_noise_ch = ch; }
    rc = enqueue_quickshift(h, h->frame.as<uint8_t>(), (int64_t)cw * 3, 0, 0, cw, ch, ratio, kernel_size, max_dist,
                            h->qs_noise.as<double>());
    if (rc) return rc;
    return finish_host_seg(h, frame, rect, h->qs_count.as<int>(), 0, labels_out, n_labels_out);
}

extern "C" int pcm_felzenszwalb(const uint8_t* frame, int H, int W, int64_t stride, const int rect[4], double scale,
                                double sigma, int min_size, const double* kernel, int kernel_radius,
                                int32_t* labels_out, int* n_labels_out) {
    if (!frame || !rect || !labels_out) return fail(PCM_E_INVALID, "pcm_felzenszwalb: NULL argument");
    if (int rc = check_rect("pcm_felzenszwalb", rect, H, W)) return rc;
    if ((long long)rect[2] * rect[3] > (1LL << 28)) return fail(PCM_E_LIMIT, "pcm_felzenszwalb: crop too large");
    if (kernel && kernel_radius < 0) return fail(PCM_E_INVALID, "pcm_felzenszwalb: kernel_radius %d", kernel_radius);
    const int n = felzenszwalb(frame, stride, rect[0], rect[1], rect[2], rect[3], scale, sigma, min_size, kernel,
                               kernel_radius, labels_out);
    if (n < 0) return fail(PCM_E_INVALID, "pcm_felzenszwalb: bad arguments");
    if (n_labels_out) *n_labels_out = n;
    return PCM_OK;
}

// the arguments of pcm_slic and its GPU variants besides the frame and a crop rect already checked with check_rect
static int check_slic_args(const char* who, const int rect[4], int n_segments, double compactness, int max_iter, int start_label,
                           const double* kernel, int kernel_radius) {
    if ((long long)rect[2] * rect[3] > (1LL << 28)) return fail(PCM_E_LIMIT, "%s: crop too large (more than 2^28 pixels)", who);
    if (n_segments < 1) return fail(PCM_E_INVALID, "%s: n_segments %d < 1", who, n_segments);
    if (!(compactness > 0)) return fail(PCM_E_INVALID, "%s: compactness must be > 0", who);
    if (max_iter < 0) return fail(PCM_E_INVALID, "%s: max_iter %d < 0", who, max_iter);
    if (start_label < 0) return fail(PCM_E_INVALID, "%s: start_label %d", who, start_label);
    if (kernel && kernel_radius < 0) return fail(PCM_E_INVALID, "%s: kernel_radius %d", who, kernel_radius);
    return PCM_OK;
}

extern "C" int pcm_slic(const uint8_t* frame, int H, int W, int64_t stride, const int rect[4], int n_segments,
                        double compactness, double sigma, const double* kernel, int kernel_radius, int max_iter,
                        int start_label, int32_t* labels_out, int* n_labels_out) {
    if (!frame || !rect || !labels_out) return fail(PCM_E_INVALID, "pcm_slic: NULL argument");
    if (int rc = check_rect("pcm_slic", rect, H, W)) return rc;
    if (int rc = check_slic_args("pcm_slic", rect, n_segments, compactness, max_iter, start_label, kernel, kernel_radius)) return rc;
    const int n = slic(frame, stride, rect[0], rect[1], rect[2], rect[3], n_segments, compactness, sigma, kernel, kernel_radius,
                       max_iter, start_label, labels_out);
    if (n < 0) return fail(PCM_E_INVALID, "pcm_slic: bad arguments (n_segments >= 1, compactness > 0, max_iter >= 0)");
    if (n_labels_out) *n_labels_out = n;
    return PCM_OK;
}

extern "C" int pcm_felzenszwalb_graph(int n_vertices, int n_edges, const int32_t* a, const int32_t* b, const double* cost,
                                      double scale, int min_size, int32_t* labels_out, int* n_labels_out) {
    if (!a || !b || !cost || !labels_out) return fail(PCM_E_INVALID, "pcm_felzenszwalb_graph: NULL argument");
    if (n_vertices <= 0 || n_vertices > (1 << 28) || n_edges < 0) return fail(PCM_E_INVALID, "pcm_felzenszwalb_graph: bad sizes");
    const int n = felzenszwalb_graph(n_vertices, n_edges, a, b, cost, scale, min_size, labels_out);
    if (n < 0) return fail(PCM_E_INVALID, "pcm_felzenszwalb_graph: vertex index out of range or negative / NaN cost");
    if (n_labels_out) *n_labels_out = n;
    return PCM_OK;
}

// ---------------------------------------------------------------------------------
// API: SLIC over-segmentation on the GPU (pcm_slic.cuh).  Same labels as pcm_slic; see DESIGN.md §10.
// ---------------------------------------------------------------------------------
// regular_grid((1, h, w), n_points) as pcm_slic.cpp's slic_grid computes it (same expressions, host code): start and step of
// the seed grid along rows and columns; false: every pixel is a seed
static bool slic_seed_grid(int h, int w, int n_points, int& start_y, int& step_y, int& start_x, int& step_x) {
    const double space = (double)h * (double)w;
    if (space <= (double)n_points) return false;
    double steps[3] = {std::pow(space / n_points, 1.0 / 3), 0, 0};
    steps[1] = steps[2] = steps[0];
    const double dims[3] = {1.0, (double)std::min(h, w), (double)std::max(h, w)};
    bool any_short = false;
    for (int d = 0; d < 3; ++d) any_short = any_short || dims[d] < steps[d];
    if (any_short) {
        for (int d = 0; d < 3; ++d) {
            steps[d] = dims[d];
            double sp = 1.0;
            for (int e = d + 1; e < 3; ++e) sp *= dims[e];
            for (int e = d + 1; e < 3; ++e) steps[e] = std::pow(sp / n_points, 1.0 / (3 - d - 1));
            bool ok = true;
            for (int e = 0; e < 3; ++e) ok = ok && dims[e] >= steps[e];
            if (ok) break;
        }
    }
    const int s_min = (int)std::floor(steps[1] / 2), s_max = (int)std::floor(steps[2] / 2);
    const int t_min = (int)std::nearbyint(steps[1]), t_max = (int)std::nearbyint(steps[2]);
    if (h <= w) { start_y = s_min; step_y = t_min; start_x = s_max; step_x = t_max; }
    else        { start_y = s_max; step_y = t_max; start_x = s_min; step_x = t_min; }
    step_y = std::max(step_y, 1); step_x = std::max(step_x, 1);
    return true;
}

static int bit_length(unsigned v) { int b = 0; while (v) { ++b; v >>= 1; } return b; }

// CUB scratch for a stable sort of n (int key, int value) pairs and an exclusive sum of n ints
static int reserve_slic_cub(pcm_handle* h, int n, size_t* bytes) {
    size_t a = 0, b = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, a, (const int*)nullptr, (int*)nullptr, (const int*)nullptr, (int*)nullptr, n));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, b, (const int*)nullptr, (int*)nullptr, n));
    *bytes = std::max(a, b);
    CUDA_TRY(h->sl_cub.reserve(*bytes));
    return PCM_OK;
}

// S5 of pcm_slic.cuh: connectivity enforcement of the centre map d_seg (w x hh) into d_labels; the largest label goes to
// sl_count.  Asynchronous.
static int enqueue_slic_connectivity(pcm_handle* h, const int32_t* d_seg, int w, int hh, long long min_size, long long max_size,
                                     int start_label, int32_t* d_labels) {
    const int n = w * hh;
    const size_t ib = (size_t)n * sizeof(int);
    cudaStream_t st = h->stream;
    for (DevBuf* b : {&h->sl_parent, &h->sl_root, &h->sl_csize, &h->sl_piece, &h->sl_psize, &h->sl_off, &h->sl_queue, &h->sl_seen,
                      &h->sl_adj, &h->sl_nxt, &h->sl_val, &h->sl_keys, &h->sl_iota, &h->sl_sidx})
        CUDA_TRY(b->reserve(ib));
    CUDA_TRY(h->sl_count.reserve(sizeof(int)));
    size_t cub_bytes = 0;
    if (int rc = reserve_slic_cub(h, n, &cub_bytes)) return rc;
    const int blocks = (int)std::min<long long>((n + SLIC_THREADS - 1) / SLIC_THREADS, (long long)h->sm_count * 16);
    int* parent = h->sl_parent.as<int>();
    int* root = h->sl_root.as<int>();
    int* csize = h->sl_csize.as<int>();
    int* piece = h->sl_piece.as<int>();
    int* psize = h->sl_psize.as<int>();
    int* off = h->sl_off.as<int>();
    int* iota = h->sl_iota.as<int>();
    slic_ccl_init_kernel<<<blocks, SLIC_THREADS, 0, st>>>(iota, n);
    CHECK_LAUNCH(h, "slic_ccl_init_kernel");
    slic_ccl_init_kernel<<<blocks, SLIC_THREADS, 0, st>>>(parent, n);
    CHECK_LAUNCH(h, "slic_ccl_init_kernel");
    slic_ccl_merge_kernel<<<blocks, SLIC_THREADS, 0, st>>>(d_seg, parent, w, hh);
    CHECK_LAUNCH(h, "slic_ccl_merge_kernel");
    CUDA_TRY(cudaMemsetAsync(csize, 0, ib, st));
    slic_ccl_flatten_kernel<<<blocks, SLIC_THREADS, 0, st>>>(parent, root, csize, n);
    CHECK_LAUNCH(h, "slic_ccl_flatten_kernel");
    CUDA_TRY(cudaMemsetAsync(psize, 0, ib, st));
    slic_piece_init_kernel<<<blocks, SLIC_THREADS, 0, st>>>(root, csize, max_size, piece, psize, n);
    CHECK_LAUNCH(h, "slic_piece_init_kernel");
    // the pixels of each component in raster order: stable sort by root; the component of root r starts at coff[r]
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(h->sl_cub.p, cub_bytes, root, h->sl_keys.as<int>(), iota, h->sl_sidx.as<int>(), n, 0,
                                             std::max(1, bit_length((unsigned)(n - 1))), st));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(h->sl_cub.p, cub_bytes, csize, off, n, st));
    slic_split_kernel<<<blocks, SLIC_THREADS, 0, st>>>(d_seg, csize, off, h->sl_sidx.as<int>(), w, hh, max_size, piece, psize,
                                                       h->sl_queue.as<int>());
    CHECK_LAUNCH(h, "slic_split_kernel");
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(h->sl_cub.p, cub_bytes, psize, off, n, st));
    CUDA_TRY(cudaMemsetAsync(h->sl_seen.p, 0, ib, st));
    slic_small_kernel<<<blocks, SLIC_THREADS, 0, st>>>(piece, psize, off, w, hh, min_size, max_size, h->sl_queue.as<int>(),
                                                       h->sl_seen.as<int>(), h->sl_adj.as<int>());
    CHECK_LAUNCH(h, "slic_small_kernel");
    slic_flag_kernel<<<blocks, SLIC_THREADS, 0, st>>>(psize, min_size, parent, n);
    CHECK_LAUNCH(h, "slic_flag_kernel");
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(h->sl_cub.p, cub_bytes, parent, off, n, st));
    slic_link_kernel<<<blocks, SLIC_THREADS, 0, st>>>(psize, off, h->sl_adj.as<int>(), min_size, start_label, h->sl_nxt.as<int>(),
                                                      h->sl_val.as<int>(), n);
    CHECK_LAUNCH(h, "slic_link_kernel");
    for (int r = bit_length((unsigned)n); r >= 0; --r) {          // a chain of at most n pieces: ceil(log2 n) + 1 rounds
        slic_jump_kernel<<<blocks, SLIC_THREADS, 0, st>>>(psize, h->sl_nxt.as<int>(), n);
        CHECK_LAUNCH(h, "slic_jump_kernel");
    }
    CUDA_TRY(cudaMemsetAsync(h->sl_count.p, 0xff, sizeof(int), st));
    slic_label_kernel<<<blocks, SLIC_THREADS, 0, st>>>(piece, h->sl_nxt.as<int>(), h->sl_val.as<int>(), d_labels, h->sl_count.as<int>(), n);
    CHECK_LAUNCH(h, "slic_label_kernel");
    return PCM_OK;
}

// The whole SLIC of the crop (cx, cy, w, hh) of a device frame into seg_labels.  Asynchronous apart from the host-side
// staging of the weights and seeds; the largest label goes to sl_count.
static int enqueue_slic(pcm_handle* h, const uint8_t* d_frame, int64_t stride, int cx, int cy, int w, int hh, int n_segments,
                        double compactness, double sigma, const double* kernel, int radius, int max_iter, int start_label) {
    const int n = w * hh;
    cudaStream_t st = h->stream;
    h->chain_tail = false;
    h->sl_w = h->sl_h = 0;
    // Gaussian weights: the caller's, or scipy's _gaussian_kernel1d computed as pcm_slic.cpp does (truncate = 4)
    std::vector<double> kw;
    if (sigma > 0 && !kernel) {
        radius = (int)(4.0 * sigma + 0.5);
        kw.resize(2 * radius + 1);
        double sum = 0;
        for (int x = -radius; x <= radius; ++x) { kw[x + radius] = std::exp(-0.5 / (sigma * sigma) * (double)(x * x)); sum += kw[x + radius]; }
        for (double& v : kw) v /= sum;
        kernel = kw.data();
    }
    if (!(sigma > 0)) radius = 0;
    // seeds on the regular grid (every pixel when there are no more pixels than segments)
    int sy = 0, ty = 1, sx = 0, tx = 1;
    const bool grid = slic_seed_grid(hh, w, n_segments, sy, ty, sx, tx);
    if (!grid) { sy = sx = 0; ty = tx = 1; }
    const int ny = sy < hh ? (hh - sy + ty - 1) / ty : 0, nx = sx < w ? (w - sx + tx - 1) / tx : 0;
    const long long K = (long long)ny * nx;
    if (K < 1) return fail(PCM_E_INVALID, "slic: no seed inside the %dx%d crop", w, hh);
    const double step = (double)std::max(1, std::max(ty, tx));
    const double spatial_weight = 1.0 / (step * step);
    const size_t nk = sigma > 0 ? (size_t)(2 * radius + 1) : 0;
    const size_t cbytes = (size_t)K * 5 * sizeof(double);
    CUDA_TRY(h->h_slic.reserve(nk * sizeof(double) + cbytes));
    double* hk = h->h_slic.as<double>();
    if (nk) memcpy(hk, kernel, nk * sizeof(double));
    double* hc = hk + nk;
    for (int a = 0; a < ny; ++a)
        for (int b = 0; b < nx; ++b) {
            double* c = hc + ((size_t)a * nx + b) * 5;
            c[0] = sy + a * ty; c[1] = sx + b * tx; c[2] = c[3] = c[4] = 0.0;
        }
    const size_t ib = (size_t)n * sizeof(int), db = (size_t)n * 3 * sizeof(double);
    CUDA_TRY(h->sl_kernel.reserve(std::max<size_t>(nk, 1) * sizeof(double)));
    CUDA_TRY(h->sl_centers.reserve(cbytes));
    CUDA_TRY(h->sl_smooth.reserve(db));
    CUDA_TRY(h->sl_tmp.reserve(db));
    CUDA_TRY(h->sl_img.reserve(db));
    CUDA_TRY(h->sl_dmin.reserve((size_t)n * sizeof(unsigned long long)));
    for (DevBuf* b : {&h->sl_best, &h->sl_nearest, &h->sl_keys, &h->sl_iota, &h->sl_sidx}) CUDA_TRY(b->reserve(ib));
    CUDA_TRY(h->sl_begin.reserve((size_t)K * sizeof(int)));
    CUDA_TRY(h->sl_end.reserve((size_t)K * sizeof(int)));
    CUDA_TRY(h->seg_labels.reserve(ib));
    size_t cub_bytes = 0;
    if (int rc = reserve_slic_cub(h, n, &cub_bytes)) return rc;
    if (nk) CUDA_TRY(cudaMemcpyAsync(h->sl_kernel.p, hk, nk * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(h->sl_centers.p, hc, cbytes, cudaMemcpyHostToDevice, st));
    h->bytes_h2d += (int64_t)(nk * sizeof(double) + cbytes);

    const int blocks = (int)std::min<long long>(((long long)n + SLIC_THREADS - 1) / SLIC_THREADS, (long long)h->sm_count * 16);
    const double* dk = h->sl_kernel.as<double>();
    double* smooth = h->sl_smooth.as<double>();
    slic_load_kernel<<<blocks, SLIC_THREADS, 0, st>>>(d_frame, stride, cx, cy, w, hh, dk, radius, sigma > 0 ? 1 : 0, smooth);
    CHECK_LAUNCH(h, "slic_load_kernel");
    if (sigma > 0) {
        slic_smooth_kernel<<<blocks, SLIC_THREADS, 0, st>>>(smooth, h->sl_tmp.as<double>(), hh, w, 0, dk, radius);
        CHECK_LAUNCH(h, "slic_smooth_kernel");
        slic_smooth_kernel<<<blocks, SLIC_THREADS, 0, st>>>(h->sl_tmp.as<double>(), smooth, hh, w, 1, dk, radius);
        CHECK_LAUNCH(h, "slic_smooth_kernel");
    }
    const double* img = h->sl_img.as<double>();
    slic_lab_kernel<<<blocks, SLIC_THREADS, 0, st>>>(smooth, h->sl_img.as<double>(), n, 1.0 / compactness);
    CHECK_LAUNCH(h, "slic_lab_kernel");

    int* nearest = h->sl_nearest.as<int>();
    int* iota = h->sl_iota.as<int>();
    double* centers = h->sl_centers.as<double>();
    CUDA_TRY(cudaMemsetAsync(nearest, 0, ib, st));
    slic_ccl_init_kernel<<<blocks, SLIC_THREADS, 0, st>>>(iota, n);
    CHECK_LAUNCH(h, "slic_ccl_init_kernel");
    const int key_bits = std::max(1, bit_length((unsigned)(K - 1)));
    for (int it = 0; it < max_iter; ++it) {
        CUDA_TRY(cudaMemsetAsync(h->sl_dmin.p, 0xff, (size_t)n * sizeof(unsigned long long), st));
        CUDA_TRY(cudaMemsetAsync(h->sl_best.p, 0x7f, ib, st));
        slic_assign_kernel<false><<<(unsigned)K, SLIC_THREADS, 0, st>>>(img, centers, hh, w, ty, tx, spatial_weight,
                                                                         h->sl_dmin.as<unsigned long long>(), h->sl_best.as<int>());
        CHECK_LAUNCH(h, "slic_assign_kernel<false>");
        slic_assign_kernel<true><<<(unsigned)K, SLIC_THREADS, 0, st>>>(img, centers, hh, w, ty, tx, spatial_weight,
                                                                        h->sl_dmin.as<unsigned long long>(), h->sl_best.as<int>());
        CHECK_LAUNCH(h, "slic_assign_kernel<true>");
        slic_settle_kernel<<<blocks, SLIC_THREADS, 0, st>>>(h->sl_best.as<int>(), nearest, n);
        CHECK_LAUNCH(h, "slic_settle_kernel");
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(h->sl_cub.p, cub_bytes, nearest, h->sl_keys.as<int>(), iota, h->sl_sidx.as<int>(), n,
                                                 0, key_bits, st));
        CUDA_TRY(cudaMemsetAsync(h->sl_begin.p, 0, (size_t)K * sizeof(int), st));
        CUDA_TRY(cudaMemsetAsync(h->sl_end.p, 0, (size_t)K * sizeof(int), st));
        slic_bounds_kernel<<<blocks, SLIC_THREADS, 0, st>>>(h->sl_keys.as<int>(), n, h->sl_begin.as<int>(), h->sl_end.as<int>());
        CHECK_LAUNCH(h, "slic_bounds_kernel");
        slic_update_kernel<<<(unsigned)((K + 127) / 128), 128, 0, st>>>(h->sl_sidx.as<int>(), h->sl_begin.as<int>(), h->sl_end.as<int>(),
                                                                         img, w, (int)K, centers);
        CHECK_LAUNCH(h, "slic_update_kernel");
    }
    // connectivity: min_size_factor 0.5, max_size_factor 3 of the requested segment size
    const double segment_size = (double)hh * (double)w / n_segments;
    const long long min_size = (long long)(0.5 * segment_size), max_size = (long long)(3 * segment_size);
    if (int rc = enqueue_slic_connectivity(h, nearest, w, hh, min_size, max_size, start_label, h->seg_labels.as<int32_t>())) return rc;
    h->sl_w = w; h->sl_h = hh;
    return PCM_OK;
}

extern "C" int pcm_slic_device(pcm_handle* h, const uint8_t* d_frame, int H, int W, int64_t stride, const int rect[4],
                               int n_segments, double compactness, double sigma, const double* kernel, int kernel_radius,
                               int max_iter, int start_label, int32_t* d_labels_out, int* n_labels_out) {
    return seg_device(h, "pcm_slic_device", d_frame, H, W, stride, rect, &pcm_handle::sl_count, 1, d_labels_out, n_labels_out, [&] {
        if (int rc = check_slic_args("pcm_slic_device", rect, n_segments, compactness, max_iter, start_label, kernel, kernel_radius))
            return rc;
        CUDA_TRY(cudaStreamSynchronize(h->stream));      // the pinned seed buffer is reused between calls
        return enqueue_slic(h, d_frame, stride, rect[0], rect[1], rect[2], rect[3], n_segments, compactness, sigma, kernel,
                            kernel_radius, max_iter, start_label);
    });
}

extern "C" int pcm_slic_device_batch(pcm_handle* h, int n, const uint8_t* d_frames, int64_t frame_bytes, const int32_t* frame_index,
                                     int H, int W, int64_t stride, const int32_t* rects, int n_segments, double compactness,
                                     double sigma, const double* kernel, int kernel_radius, int max_iter, int start_label,
                                     int32_t* d_labels_out, const int64_t* label_offsets, int32_t* n_labels_out) {
    return seg_device_batch(h, "pcm_slic_device_batch", n, d_frames, frame_bytes, frame_index, rects, d_labels_out, label_offsets,
                            n_labels_out, [&](const uint8_t* d_frame, const int rect[4], int32_t* d_labels, int* count) {
                                return pcm_slic_device(h, d_frame, H, W, stride, rect, n_segments, compactness, sigma, kernel,
                                                       kernel_radius, max_iter, start_label, d_labels, count);
                            });
}

extern "C" int pcm_slic_gpu(pcm_handle* h, const uint8_t* frame, int H, int W, int64_t stride, const int rect[4], int n_segments,
                            double compactness, double sigma, const double* kernel, int kernel_radius, int max_iter,
                            int start_label, int32_t* labels_out, int* n_labels_out) {
    int rc = begin_seg(h, "pcm_slic_gpu", frame, H, W, stride, rect);
    if (rc) return rc;
    if ((rc = check_slic_args("pcm_slic_gpu", rect, n_segments, compactness, max_iter, start_label, kernel, kernel_radius))) return rc;
    if ((rc = stage_crop(h, "pcm_slic_gpu", frame, stride, rect, 0, [](int) { return cudaSuccess; }))) return rc;
    rc = enqueue_slic(h, h->frame.as<uint8_t>(), (int64_t)rect[2] * 3, 0, 0, rect[2], rect[3], n_segments, compactness, sigma, kernel,
                      kernel_radius, max_iter, start_label);
    if (rc) return rc;
    return finish_host_seg(h, frame, rect, h->sl_count.as<int>(), 1, labels_out, n_labels_out);
}

extern "C" int pcm_slic_connectivity(pcm_handle* h, const int32_t* nearest, int width, int height, long long min_size,
                                     long long max_size, int start_label, int32_t* labels_out, int* n_labels_out) {
    if (!h || !nearest || !labels_out) return fail(PCM_E_INVALID, "pcm_slic_connectivity: NULL argument");
    if (width <= 0 || height <= 0 || (long long)width * height > (1LL << 28))
        return fail(PCM_E_INVALID, "pcm_slic_connectivity: bad size %dx%d", width, height);
    if (start_label < 0) return fail(PCM_E_INVALID, "pcm_slic_connectivity: start_label %d", start_label);
    CUDA_TRY(cudaSetDevice(h->device));
    const size_t ib = (size_t)width * height * sizeof(int32_t);
    cudaStream_t st = h->stream;
    h->chain_tail = false;
    CUDA_TRY(h->sl_best.reserve(ib));
    CUDA_TRY(h->sl_labels.reserve(ib));
    CUDA_TRY(cudaMemcpyAsync(h->sl_best.p, nearest, ib, cudaMemcpyHostToDevice, st));
    int rc = enqueue_slic_connectivity(h, h->sl_best.as<int32_t>(), width, height, min_size, max_size, start_label,
                                       h->sl_labels.as<int32_t>());
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(labels_out, h->sl_labels.p, ib, cudaMemcpyDeviceToHost, st));
    int count = 0;
    if ((rc = read_seg_count(h, h->sl_count.as<int>(), 1, &count))) return rc;
    if (n_labels_out) *n_labels_out = count;
    return PCM_OK;
}

extern "C" int pcm_slic_debug_last(pcm_handle* h, double* smoothed, double* image, int32_t* nearest) {
    if (!h) return fail(PCM_E_INVALID, "pcm_slic_debug_last: NULL handle");
    if (!h->sl_w) return fail(PCM_E_STATE, "pcm_slic_debug_last: no SLIC on this handle yet");
    CUDA_TRY(cudaSetDevice(h->device));
    const size_t n = (size_t)h->sl_w * h->sl_h;
    cudaStream_t st = h->stream;
    if (smoothed) CUDA_TRY(cudaMemcpyAsync(smoothed, h->sl_smooth.p, 3 * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (image) CUDA_TRY(cudaMemcpyAsync(image, h->sl_img.p, 3 * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (nearest) CUDA_TRY(cudaMemcpyAsync(nearest, h->sl_nearest.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return PCM_OK;
}

// ---------------------------------------------------------------------------------
// API: SIFT-match prior on the device (SURVEY.md §8 f-2)
// ---------------------------------------------------------------------------------
extern "C" int pcm_prior_device(pcm_handle* h, const float* d_pts_prev, const uint8_t* d_des_prev, int n_prev,
                                const uint8_t* d_prev_mask, int64_t prev_mask_stride, int prev_w, int prev_h,
                                const float* d_pts, const uint8_t* d_des, int n_cur, const int32_t* d_labels, int crop_w,
                                int crop_h, int n_labels, float* d_priors) {
    if (!h || !d_labels || !d_priors) return fail(PCM_E_INVALID, "pcm_prior_device: NULL argument");
    if (n_prev < 0 || n_cur < 0 || n_labels < 1 || crop_w < 1 || crop_h < 1 || prev_w < 1 || prev_h < 1)
        return fail(PCM_E_INVALID, "pcm_prior_device: bad size");
    if (n_prev > 0 && (!d_pts_prev || !d_des_prev || !d_prev_mask)) return fail(PCM_E_INVALID, "pcm_prior_device: NULL argument");
    if (n_cur > 0 && (!d_pts || !d_des)) return fail(PCM_E_INVALID, "pcm_prior_device: NULL argument");
    if (((uintptr_t)d_des_prev | (uintptr_t)d_des) & 15) return fail(PCM_E_INVALID, "pcm_prior_device: descriptors must be 16-byte aligned");
    CUDA_TRY(cudaSetDevice(h->device));
    h->chain_tail = false;
    cudaStream_t st = h->stream;
    const size_t m1 = (size_t)std::max(n_prev, 1);
    CUDA_TRY(h->prior_scratch.reserve(m1 * (2 * sizeof(double) + 2 * sizeof(int))));
    char* sb = h->prior_scratch.as<char>();
    PriorArgs a{};
    a.pts1 = d_pts_prev; a.des1 = d_des_prev; a.m1 = n_prev;
    a.prev_mask = d_prev_mask; a.prev_stride = prev_mask_stride; a.prev_w = prev_w; a.prev_h = prev_h;
    a.pts2 = d_pts; a.des2 = d_des; a.m2 = n_cur;
    a.labels = d_labels; a.cw = crop_w; a.ch = crop_h; a.n_labels = n_labels; a.priors = d_priors;
    a.q_dist = reinterpret_cast<double*>(sb);
    a.g_dist = a.q_dist + m1;
    a.q_j = reinterpret_cast<int*>(a.g_dist + m1);
    a.g_j = a.q_j + m1;
    if (n_prev > 0) {
        prior_match_kernel<<<(n_prev + 7) / 8, 256, 0, st>>>(a);
        CHECK_LAUNCH(h, "prior_match_kernel");
    }
    prior_finish_kernel<<<1, 1024, 0, st>>>(a);
    CHECK_LAUNCH(h, "prior_finish_kernel");
    return PCM_OK;
}

static_assert(sizeof(pcm_frame_job) == 200 && offsetof(pcm_frame_job, d_pts) == 128 && offsetof(pcm_frame_job, d_counts) == 192,
              "pcm_frame_job layout is part of the ABI (pcm/capi.py: FrameJob)");

extern "C" int pcm_run_frames(pcm_handle* h, int frame_h, int frame_w, int64_t frame_stride, uint8_t* d_mask,
                              int64_t mask_row_stride, const pcm_frame_job* jobs, int n_jobs) {
    if (!h || !d_mask || (!jobs && n_jobs > 0)) return fail(PCM_E_INVALID, "pcm_run_frames: NULL argument");
    if (n_jobs < 0 || frame_h <= 0 || frame_w <= 0 || mask_row_stride < frame_w) return fail(PCM_E_INVALID, "pcm_run_frames: bad size");
    CUDA_TRY(cudaSetDevice(h->device));
    // At most `ahead` frames are in flight on the stream: the thread waits (blocking-sync event, CPU yielded) for frame
    // k - ahead before it enqueues frame k.  Without the limit a long sequence fills the stream's launch queue and the
    // thread then blocks INSIDE a launch call, which serialises the launches of the other sequence threads of the
    // process (the sweep runs 8 - 16 of them, each on its own stream).  Measured (256-sequence sweep, 16 threads), in
    // sequences/s: no limit -> 52-69, 8 -> 73-81, 32 -> 76-78.
    constexpr int ahead = 8;
    if ((int)h->ahead_events.size() < ahead) {
        const size_t old = h->ahead_events.size();
        h->ahead_events.resize((size_t)ahead, nullptr);
        for (size_t i = old; i < h->ahead_events.size(); ++i)
            CUDA_TRY(cudaEventCreateWithFlags(&h->ahead_events[i], cudaEventDisableTiming | cudaEventBlockingSync));
    }
    for (int k = 0; k < n_jobs; ++k) {
        const pcm_frame_job& j = jobs[k];
        int rc;
        if (k >= ahead) CUDA_TRY(cudaEventSynchronize(h->ahead_events[k % ahead]));
        if (j.d_priors_out) {
            rc = pcm_prior_device(h, j.d_pts_prev, j.d_des_prev, j.n_prev,
                                  d_mask + (int64_t)j.prev_rect[1] * mask_row_stride + j.prev_rect[0], mask_row_stride,
                                  j.prev_rect[2], j.prev_rect[3], j.d_pts, j.d_des, j.n_cur, j.d_labels, j.rect[2], j.rect[3],
                                  j.n_labels, j.d_priors_out);
            if (rc) return rc;
        }
        if (j.clear_mask == 1) {
            CUDA_TRY(cudaMemsetAsync(d_mask, 0, (size_t)mask_row_stride * frame_h, h->stream));
            h->chain_tail = false;
        }
        const int rect[4] = {j.rect[0], j.rect[1], j.rect[2], j.rect[3]};
        rc = pcm_update_device(h, j.d_frame, frame_h, frame_w, frame_stride, rect, j.d_labels, j.n_labels,
                               j.d_priors_out ? j.d_priors_out : j.d_priors, &j.params, d_mask, mask_row_stride);
        if (rc) return rc;
        if (j.d_truth) {
            rc = enqueue_iou(h, d_mask, mask_row_stride, j.d_truth, j.truth_stride, j.truth_channels, frame_h, frame_w, j.d_counts,
                             j.clear_mask == 2 ? rect : nullptr);
            if (rc) return rc;
        }
        if (k + ahead < n_jobs) CUDA_TRY(cudaEventRecord(h->ahead_events[k % ahead], h->stream));
    }
    return PCM_OK;
}

// ---------------------------------------------------------------------------------
// API: training (SURVEY.md §8 f-3): the forest of addModel, grown on the GPU
// ---------------------------------------------------------------------------------
static int upload_fit_rows(pcm_handle* h, const int16_t* X, const uint8_t* y, int n_rows, int n_features, long long rows_id) {
    cudaStream_t st = h->stream;
    const size_t n = (size_t)n_rows;
    const long long n_pad = ((long long)n_rows + 63) / 64 * 64;
    h->fit_rows_id = 0;
    CUDA_TRY(h->fit_x.reserve(n * n_features * sizeof(int16_t)));
    CUDA_TRY(h->fit_xt.reserve((size_t)n_pad * n_features * sizeof(int16_t)));
    CUDA_TRY(h->fit_y.reserve(n));
    CUDA_TRY(cudaMemcpyAsync(h->fit_x.p, X, n * n_features * sizeof(int16_t), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(h->fit_y.p, y, n, cudaMemcpyHostToDevice, st));
    fit_transpose_kernel<<<dim3((n_rows + 31) / 32, (n_features + 31) / 32), dim3(32, 8), 0, st>>>(
        h->fit_x.as<int16_t>(), n_rows, n_features, h->fit_xt.as<int16_t>(), n_pad);
    CHECK_LAUNCH(h, "fit_transpose_kernel");
    h->fit_rows_id = rows_id;
    h->fit_n = n_rows; h->fit_F = n_features;
    return PCM_OK;
}

static int check_fit_rows(pcm_handle* h, const char* who, const uint8_t* y, int n_rows, int n_features) {
    if (!h || !y) return fail(PCM_E_INVALID, "%s: NULL argument", who);
    if (n_rows < 1 || n_rows >= (1 << 24)) return fail(PCM_E_LIMIT, "%s: n_rows %d outside [1, 2^24)", who, n_rows);
    if (n_features < 1 || n_features > FIT_MAX_FEATURES)
        return fail(PCM_E_LIMIT, "%s: n_features %d outside [1, %d]", who, n_features, FIT_MAX_FEATURES);
    return PCM_OK;
}

extern "C" int pcm_fit_rows(pcm_handle* h, const int16_t* X, const uint8_t* y, int n_rows, int n_features, long long rows_id) {
    int rc = check_fit_rows(h, "pcm_fit_rows", y, n_rows, n_features);
    if (rc) return rc;
    if (!X) return fail(PCM_E_INVALID, "pcm_fit_rows: NULL argument");
    CUDA_TRY(cudaSetDevice(h->device));
    h->chain_tail = false;
    return upload_fit_rows(h, X, y, n_rows, n_features, rows_id);
}

extern "C" int pcm_fit_forest(pcm_handle* h, const int16_t* X, const uint8_t* y, int n_rows, int n_features,
                              long long rows_id, int n_trees, int max_depth, int max_features, const uint8_t* counts,
                              const uint32_t* rand_states, int node_capacity, int32_t* node_count, int32_t* feature,
                              double* threshold, int32_t* left, int32_t* right, double* value1, int32_t* n_node_samples) {
    int rc = check_fit_rows(h, "pcm_fit_forest", y, n_rows, n_features);
    if (rc) return rc;
    if (!counts || !rand_states || !node_count || !feature || !threshold || !left || !right || !value1)
        return fail(PCM_E_INVALID, "pcm_fit_forest: NULL argument");
    if (n_trees < 1) return fail(PCM_E_INVALID, "pcm_fit_forest: n_trees %d", n_trees);
    if (max_depth < 0 || max_depth > FIT_MAX_DEPTH)
        return fail(PCM_E_LIMIT, "pcm_fit_forest: max_depth %d outside [0, %d]", max_depth, FIT_MAX_DEPTH);
    if (max_features < 1 || max_features > n_features) return fail(PCM_E_INVALID, "pcm_fit_forest: max_features %d", max_features);
    if (node_capacity < 1) return fail(PCM_E_INVALID, "pcm_fit_forest: node_capacity %d", node_capacity);
    const bool resident = !X;
    if (resident && (rows_id == 0 || rows_id != h->fit_rows_id || n_rows != h->fit_n || n_features != h->fit_F))
        return fail(PCM_E_STATE, "pcm_fit_forest: X == NULL needs the rows of a previous call with the same rows_id");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    h->chain_tail = false;
    const size_t n = (size_t)n_rows, T = (size_t)n_trees, cap = (size_t)node_capacity;
    const long long n_pad = ((long long)n_rows + 63) / 64 * 64;
    for (size_t i = 0; i < T * n; ++i)
        if (counts[i] > 127) return fail(PCM_E_LIMIT, "pcm_fit_forest: bootstrap count %d > 127", (int)counts[i]);
    if (!resident) {
        rc = upload_fit_rows(h, X, y, n_rows, n_features, rows_id);
        if (rc) return rc;
    }
    CUDA_TRY(h->fit_counts.reserve(T * n));
    CUDA_TRY(h->fit_rand.reserve(T * sizeof(uint32_t)));
    CUDA_TRY(h->fit_samples.reserve(T * n * sizeof(uint32_t)));
    CUDA_TRY(h->fit_tmp.reserve(T * n * sizeof(uint32_t)));
    // outputs: [feature i32 | left i32 | right i32 | n_node_samples i32 | node_count i32 (T)] [threshold f64 | value1 f64]
    const size_t o_feat = 0, o_left = o_feat + 4 * T * cap, o_right = o_left + 4 * T * cap, o_nns = o_right + 4 * T * cap,
                 o_cnt = o_nns + 4 * T * cap, o_thr = (o_cnt + 4 * T + 7) / 8 * 8, o_val = o_thr + 8 * T * cap,
                 o_end = o_val + 8 * T * cap;
    CUDA_TRY(h->fit_out.reserve(o_end));
    CUDA_TRY(cudaMemcpyAsync(h->fit_counts.p, counts, T * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(h->fit_rand.p, rand_states, T * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    char* ob = h->fit_out.as<char>();
    FitArgs a{};
    a.Xt = h->fit_xt.as<int16_t>(); a.n_pad = n_pad;
    a.y = h->fit_y.as<uint8_t>(); a.counts = h->fit_counts.as<uint8_t>(); a.rand_state = h->fit_rand.as<uint32_t>();
    a.n = n_rows; a.F = n_features; a.max_depth = max_depth; a.max_features = max_features; a.cap = node_capacity;
    a.samples = h->fit_samples.as<uint32_t>(); a.tmp = h->fit_tmp.as<uint32_t>();
    a.feature = reinterpret_cast<int32_t*>(ob + o_feat); a.left = reinterpret_cast<int32_t*>(ob + o_left);
    a.right = reinterpret_cast<int32_t*>(ob + o_right); a.n_node_samples = reinterpret_cast<int32_t*>(ob + o_nns);
    a.node_count = reinterpret_cast<int32_t*>(ob + o_cnt);
    a.threshold = reinterpret_cast<double*>(ob + o_thr); a.value1 = reinterpret_cast<double*>(ob + o_val);
    forest_fit_kernel<<<n_trees, FIT_THREADS, 0, st>>>(a);
    CHECK_LAUNCH(h, "forest_fit_kernel");
    CUDA_TRY(cudaMemcpyAsync(feature, ob + o_feat, 4 * T * cap, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(left, ob + o_left, 4 * T * cap, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(right, ob + o_right, 4 * T * cap, cudaMemcpyDeviceToHost, st));
    if (n_node_samples) CUDA_TRY(cudaMemcpyAsync(n_node_samples, ob + o_nns, 4 * T * cap, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(node_count, ob + o_cnt, 4 * T, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(threshold, ob + o_thr, 8 * T * cap, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(value1, ob + o_val, 8 * T * cap, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    for (int t = 0; t < n_trees; ++t)
        if (node_count[t] < 0) return fail(PCM_E_LIMIT, "pcm_fit_forest: tree %d needs more than %d nodes", t, node_capacity);
    return PCM_OK;
}

extern "C" int pcm_pca_moments(pcm_handle* h, long long rows_id, double* gram, double* sums, int64_t* n_class1) {
    if (!h || !gram || !sums || !n_class1) return fail(PCM_E_INVALID, "pcm_pca_moments: NULL argument");
    if (rows_id == 0 || rows_id != h->fit_rows_id) return fail(PCM_E_STATE, "pcm_pca_moments: rows %lld are not resident", rows_id);
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    h->chain_tail = false;
    const int F = h->fit_F, n = h->fit_n;
    const long long n_pad = ((long long)n + 63) / 64 * 64;
    const size_t gb = sizeof(double) * (size_t)F * F, sb = sizeof(double) * (size_t)F;
    CUDA_TRY(h->fit_out.reserve(gb + sb + 8));
    char* ob = h->fit_out.as<char>();
    const int tiles = (F + 31) / 32;
    pca_gram_kernel<<<dim3(tiles, tiles), 256, 0, st>>>(h->fit_xt.as<int16_t>(), n_pad, h->fit_y.as<uint8_t>(), n, F,
                                                       reinterpret_cast<double*>(ob), reinterpret_cast<double*>(ob + gb),
                                                       reinterpret_cast<unsigned long long*>(ob + gb + sb));
    CHECK_LAUNCH(h, "pca_gram_kernel");
    CUDA_TRY(cudaMemcpyAsync(gram, ob, gb, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(sums, ob + gb, sb, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(n_class1, ob + gb + sb, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return PCM_OK;
}

extern "C" int pcm_pca_residuals_k(pcm_handle* h, long long rows_id, const double* mean, const double* components,
                                   int n_components, double* err) {
    if (!h || !mean || !components || !err) return fail(PCM_E_INVALID, "pcm_pca_residuals_k: NULL argument");
    if (n_components < 1) return fail(PCM_E_INVALID, "pcm_pca_residuals_k: n_components %d < 1", n_components);
    if (n_components > PCM_MAX_PCA_COMPONENTS)
        return fail(PCM_E_LIMIT, "pcm_pca_residuals_k: n_components %d > PCM_MAX_PCA_COMPONENTS (%d)", n_components,
                    PCM_MAX_PCA_COMPONENTS);
    if (rows_id == 0 || rows_id != h->fit_rows_id) return fail(PCM_E_STATE, "pcm_pca_residuals_k: rows %lld are not resident", rows_id);
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    h->chain_tail = false;
    const int F = h->fit_F, n = h->fit_n, k = n_components;
    const long long n_pad = ((long long)n + 63) / 64 * 64;
    const size_t fb = sizeof(double) * (size_t)F, cb = fb * k, eb = sizeof(double) * (size_t)n;
    CUDA_TRY(h->fit_out.reserve(cb + fb + eb));
    char* ob = h->fit_out.as<char>();
    CUDA_TRY(cudaMemcpyAsync(ob, components, cb, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ob + cb, mean, fb, cudaMemcpyHostToDevice, st));
    const size_t smem = cb + fb;                       // components | mean
    if ((long long)smem > h->max_smem_optin)
        return fail(PCM_E_LIMIT, "pcm_pca_residuals_k: %d x %d components need %zu B of shared memory", k, F, smem);
    pca_residual_kernels[k - 1]<<<(n + 255) / 256, 256, smem, st>>>(h->fit_xt.as<int16_t>(), n_pad, n, F, reinterpret_cast<double*>(ob + cb),
                                                     reinterpret_cast<double*>(ob), reinterpret_cast<double*>(ob + cb + fb));
    CHECK_LAUNCH(h, "pca_residual_kernel");
    CUDA_TRY(cudaMemcpyAsync(err, ob + cb + fb, eb, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return PCM_OK;
}

extern "C" int pcm_pca_residuals(pcm_handle* h, long long rows_id, const double* mean, const double* component, double* err) {
    if (!h || !mean || !component || !err) return fail(PCM_E_INVALID, "pcm_pca_residuals: NULL argument");
    return pcm_pca_residuals_k(h, rows_id, mean, component, 1, err);
}

// ---------------------------------------------------------------------------------
// API: parity taps
// ---------------------------------------------------------------------------------
extern "C" int pcm_convert(pcm_handle* h, const uint8_t* bgr, int height, int width, int64_t stride, int space,
                           uint8_t* out, int64_t out_stride) {
    if (!h || !bgr || !out) return fail(PCM_E_INVALID, "pcm_convert: NULL argument");
    if (space < 0 || space > 2) return fail(PCM_E_INVALID, "pcm_convert: bad space %d", space);
    if (height <= 0 || width <= 0) return fail(PCM_E_INVALID, "pcm_convert: bad size");
    CUDA_TRY(cudaSetDevice(h->device));
    const size_t bytes = (size_t)height * width * 3;
    h->chain_tail = false;
    DevBuf in, o;
    CUDA_TRY(in.reserve(bytes));
    CUDA_TRY(o.reserve(bytes));
    CUDA_TRY(cudaMemcpy2DAsync(in.p, (size_t)width * 3, bgr, stride, (size_t)width * 3, height, cudaMemcpyHostToDevice, h->stream));
    const int blocks = (int)std::min<size_t>(((size_t)height * width + 255) / 256, (size_t)h->sm_count * 16);
    convert_kernel<<<blocks, 256, 0, h->stream>>>(in.as<uint8_t>(), (long long)width * 3, height, width, space,
                                                  h->d_tables, o.as<uint8_t>(), (long long)width * 3);
    CHECK_LAUNCH(h, "convert_kernel");
    CUDA_TRY(cudaMemcpy2DAsync(out, out_stride, o.p, (size_t)width * 3, (size_t)width * 3, height, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return PCM_OK;
}

extern "C" int pcm_gather_features(pcm_handle* h, const uint8_t* frame, int H, int W, int64_t stride, const int rect[4],
                                   int16_t* X) {
    if (!h || !frame || !rect || !X) return fail(PCM_E_INVALID, "pcm_gather_features: NULL argument");
    if (!h->features_set) return fail(PCM_E_STATE, "pcm_gather_features: call pcm_set_features first");
    if (int rc = check_rect("pcm_gather_features", rect, H, W)) return rc;
    CUDA_TRY(cudaSetDevice(h->device));
    const int cw = rect[2], ch = rect[3];
    const size_t npx = (size_t)cw * ch, xbytes = npx * h->geom.F * sizeof(int16_t);
    h->chain_tail = false;
    DevBuf in, o;
    CUDA_TRY(in.reserve(npx * 3));
    CUDA_TRY(o.reserve(xbytes));
    CUDA_TRY(cudaMemcpy2DAsync(in.p, (size_t)cw * 3, frame + (size_t)rect[1] * stride + (size_t)rect[0] * 3, stride,
                               (size_t)cw * 3, ch, cudaMemcpyHostToDevice, h->stream));
    const size_t work = npx * h->geom.K;
    const int blocks = (int)std::min<size_t>((work + 255) / 256, (size_t)h->sm_count * 16);
    gather_kernel<<<blocks, 256, 0, h->stream>>>(in.as<uint8_t>(), (long long)cw * 3, 0, 0, cw, ch, h->geom, h->d_tables,
                                                 o.as<int16_t>());
    CHECK_LAUNCH(h, "gather_kernel");
    CUDA_TRY(cudaMemcpyAsync(X, o.p, xbytes, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return PCM_OK;
}

extern "C" int pcm_debug_last(pcm_handle* h, double* p1, double* sa, float* scores, int64_t* areas, uint8_t* pre,
                              int32_t* n_exact) {
    if (!h) return fail(PCM_E_INVALID, "pcm_debug_last: NULL handle");
    if (!h->last_valid) return fail(PCM_E_STATE, "pcm_debug_last: no update to report");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    const size_t npx = (size_t)h->last_cw * h->last_ch;
    const int S = h->last_S;
    const SegLayout sl = seg_layout(S);
    if ((p1 || sa) && !h->last_maps)
        return fail(PCM_E_STATE, "pcm_debug_last: the per-pixel maps are not kept (call pcm_set_debug(h, 1) first)");
    if (p1) CUDA_TRY(cudaMemcpy(p1, h->p1.p, npx * sizeof(double), cudaMemcpyDeviceToHost));
    if (sa) {
        if (h->last_novelty) CUDA_TRY(cudaMemcpy(sa, h->sa.p, npx * sizeof(double), cudaMemcpyDeviceToHost));
        else memset(sa, 0, npx * sizeof(double));
    }
    if (scores) CUDA_TRY(cudaMemcpy(scores, h->scores.p, sizeof(float) * (size_t)S, cudaMemcpyDeviceToHost));
    if (areas) {
        std::vector<int> tmp(S);
        CUDA_TRY(cudaMemcpy(tmp.data(), h->seg.as<char>() + sl.area, sizeof(int) * (size_t)S, cudaMemcpyDeviceToHost));
        for (int i = 0; i < S; ++i) areas[i] = tmp[i];
    }
    if (pre) {
        if (!h->last_pre) return fail(PCM_E_STATE, "pcm_debug_last: pre-dilation map not kept (call pcm_set_debug(h, 1) first)");
        CUDA_TRY(cudaMemcpy(pre, h->pre.p, npx, cudaMemcpyDeviceToHost));
    }
    if (n_exact) {
        int v = 0;
        CUDA_TRY(cudaMemcpy(&v, h->seg.as<char>() + sl.nflag, sizeof(int), cudaMemcpyDeviceToHost));
        *n_exact = v;
    }
    return PCM_OK;
}

extern "C" int pcm_set_debug(pcm_handle* h, int on) {
    if (!h) return fail(PCM_E_INVALID, "pcm_set_debug: NULL handle");
    h->keep_pre = (on & 1) != 0;
    h->force_exact = (on & 2) != 0;
    return PCM_OK;
}

extern "C" int pcm_debug_tables(pcm_handle* h, uint16_t* gamma, uint16_t* cbrt_tab, int32_t* sdiv, int32_t* hdiv) {
    if (!h) return fail(PCM_E_INVALID, "pcm_debug_tables: NULL handle");
    ColorTables t;
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaMemcpy(&t, h->d_tables, sizeof t, cudaMemcpyDeviceToHost));
    if (gamma) memcpy(gamma, t.gamma, sizeof t.gamma);
    if (cbrt_tab) memcpy(cbrt_tab, t.cbrt_tab, sizeof(uint16_t) * LAB_CBRT_SIZE);
    if (sdiv) memcpy(sdiv, t.sdiv, sizeof t.sdiv);
    if (hdiv) memcpy(hdiv, t.hdiv, sizeof t.hdiv);
    return PCM_OK;
}

extern "C" int64_t pcm_launch_count(const pcm_handle* h) { return h ? h->launches : 0; }

extern "C" int pcm_set_label_cache(pcm_handle* h, int on) {
    if (!h) return fail(PCM_E_INVALID, "pcm_set_label_cache: NULL handle");
    h->label_cache_on = on != 0;
    return PCM_OK;
}

extern "C" int pcm_transfer_bytes(const pcm_handle* h, int64_t out[2]) {
    if (!h || !out) return fail(PCM_E_INVALID, "pcm_transfer_bytes: NULL argument");
    out[0] = h->bytes_h2d.load();
    out[1] = h->bytes_d2h.load();
    return PCM_OK;
}

extern "C" int pcm_profile_enable(pcm_handle* h, int on) {
    if (!h) return fail(PCM_E_INVALID, "pcm_profile_enable: NULL handle");
    h->profiling = on != 0;
    return PCM_OK;
}

extern "C" int pcm_profile_read(pcm_handle* h, double* ms_sum, int64_t* count, int n, int reset) {
    if (!h) return fail(PCM_E_INVALID, "pcm_profile_read: NULL handle");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    for (auto& t : h->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) { h->prof_ms[t.id] += ms; h->prof_n[t.id]++; }
        h->free_events.push_back(t.a);
        h->free_events.push_back(t.b);
    }
    h->pending.clear();
    for (int i = 0; i < n && i < PCM_NUM_KERNELS; ++i) {
        if (ms_sum) ms_sum[i] = h->prof_ms[i];
        if (count) count[i] = h->prof_n[i];
    }
    if (reset)
        for (int i = 0; i < PCM_NUM_KERNELS; ++i) { h->prof_ms[i] = 0; h->prof_n[i] = 0; }
    return PCM_OK;
}
