// C ABI of the decoder library (include/og_decoder.h): handle, buffer management,
// stream-ordered composition of the kernels, host staging.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <vector>

#include "og_common.cuh"

namespace og {

static thread_local char g_error[1024] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

}  // namespace og

using namespace og;

namespace {

template <typename T>
struct DevBuf {
    T *ptr = nullptr;
    size_t cap = 0;    // elements
    int ensure(size_t need) {
        if (need <= cap) return OG_OK;
        if (ptr) OG_CUDA_TRY(cudaFree(ptr));
        ptr = nullptr;
        cap = 0;
        const size_t grow = need + need / 4;
        OG_CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&ptr), grow * sizeof(T)));
        cap = grow;
        return OG_OK;
    }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
    }
};

}  // namespace

constexpr int kSlots = OG_MAX_IN_FLIGHT;   // decode calls that may be in flight before a fetch
constexpr int kMaxChunks = 4;      // image ranges of one host-API call (copy / decode pipeline)
constexpr int kGraphsPerSlot = 4;  // captured device-path chains a result slot keeps
// start, after prep, K1 pass 1 | select start, select = K2 start, K2, K3, end (see mark())
constexpr int kStageEvents = 8;

struct K1Fused {
    MapView hmp;            // network-resolution heat maps (n or 2n images)
    int h, w, scale;
    bool cubic, flip;
};

// What a fused decode call ran on, kept until its result is fetched: og_fetch_result materialises
// and selects the planes whose candidate lists overflowed from `k1`, then runs K2 / K3 again.
struct CallCtx {
    K1Fused k1;
    OffsetSource src;
    FlipTablesDev ft;
    int H, W;               // full-resolution size
    LimbExtras extras;      // optional heads sampled by K2 (vector_nd == 0: none)
};

// What identifies a captured decode chain: replaying the graph is only valid for the same
// inputs, shapes, flags and slot buffers.
struct GraphKey {
    const void *hmp, *off;
    int dtype;
    size_t hmp_image_stride, off_image_stride;
    size_t hmp_plane_stride, hmp_pixel_stride, off_plane_stride, off_pixel_stride;   // planar or channels-last
    int n, hgt, w, stride, mode, flip, coco;
    uint64_t tables_version, buffers_version;
    MapView scale, jitter;                  // optional heads (og_decode_features_heads_dev_strided)
    int vector_nd, use_jitter;
    static bool same_view(const MapView &a, const MapView &b) {
        return a.ptr == b.ptr && a.dtype == b.dtype && a.image_stride == b.image_stride &&
               a.plane_stride == b.plane_stride && a.pixel_stride == b.pixel_stride;
    }
    bool operator==(const GraphKey &o) const {
        return hmp == o.hmp && off == o.off && dtype == o.dtype && coco == o.coco && hmp_image_stride == o.hmp_image_stride &&
               same_view(scale, o.scale) && same_view(jitter, o.jitter) && vector_nd == o.vector_nd &&
               use_jitter == o.use_jitter &&
               off_image_stride == o.off_image_stride && hmp_plane_stride == o.hmp_plane_stride &&
               hmp_pixel_stride == o.hmp_pixel_stride && off_plane_stride == o.off_plane_stride &&
               off_pixel_stride == o.off_pixel_stride && n == o.n && hgt == o.hgt && w == o.w &&
               stride == o.stride && mode == o.mode && flip == o.flip &&
               tables_version == o.tables_version && buffers_version == o.buffers_version;
    }
};

// K2 -> K3 hand-over and K3's tables
struct GroupScratch {
    DevBuf<int32_t> prep, cnt, redo;
    DevBuf<float4> rec;
    DevBuf<float> slab;
    void release() {
        prep.release();
        cnt.release();
        redo.release();
        rec.release();
        slab.release();
    }
};

// Everything that belongs to ONE decode call until its result has been fetched.  Calls in
// flight share nothing but the read-only configuration, so they overlap freely: each slot
// has its own stream, scratch and result buffer.
struct ResultSlot {
    // result: [meta int32: offset[n], count[n], overflow flag, -][pose rows float], pinned and
    // mapped — K3 writes the rows of every person straight into host memory (posted PCIe
    // writes from its epilogue), so there is no device copy of the poses and no D2H memcpy
    unsigned char *out_host = nullptr;
    unsigned char *out_dev = nullptr;   // the same memory as the device addresses it
    size_t out_cap = 0;
    DevBuf<int32_t> total;              // K3's row allocator
    double *frames_host = nullptr;      // [n][4] image frames of the call (pinned, mapped), see og_set_frames
    double *frames_dev = nullptr;
    int frames_cap = 0;
    bool emit_coco = false;             // this call also writes back-projected result rows
    DevBuf<float> in_hmp, in_off;       // staged network-resolution inputs (host API)
    DevBuf<float> det_score;            // K1 output
    DevBuf<int32_t> det_index;
    DevBuf<int32_t> det_count;
    DevBuf<uint32_t> cand_count;        // K1 pass 1 -> pass 2 hand-over; zero between calls
    DevBuf<uint64_t> cand_keys;
    DevBuf<uint8_t> tile_flag;          // fused K1 scratch: one flag per work block, zero between calls
    // the active-block counter, 3 spare ints, then the [blocks] int4 work list: the counter keeps its
    // place whatever the geometry of the call, so the select pass that zeroes it leaves it zero for
    // the next call even when that call lists a different number of blocks
    DevBuf<int32_t> tile_list;
    DevBuf<float> nhwc_heat;            // channels-last calls: the scan's flip-fused planar heat maps [n][C][h][w]
    DevBuf<float> limbs;                // K2 output
    GroupScratch group;
    cudaStream_t work = nullptr;        // high priority: K2 -> K3 of every call, the whole chain on the device path
    cudaEvent_t k1_done[kMaxChunks] = {nullptr};
    cudaEvent_t copied[kMaxChunks] = {nullptr};
    cudaEvent_t call_start = nullptr;
    cudaEvent_t done = nullptr;
    cudaEvent_t ev[kStageEvents] = {nullptr};
    // device-path chains of this slot, replayed while their key matches; a few per slot, so a
    // caller that rotates through a ring of input buffers still replays (least recently used
    // entry is re-captured)
    cudaGraphExec_t graph[kGraphsPerSlot] = {nullptr};
    GraphKey key[kGraphsPerSlot] = {};
    uint64_t graph_used[kGraphsPerSlot] = {0};
    uint64_t buffers_version = 1;       // bumped whenever a buffer of the slot moves
    cudaStream_t stream = nullptr;      // the caller's stream of the call
    int n = 0;
    size_t meta_bytes = 0;
    int capacity_rows = 0;
    bool pending = false;
    bool fused = false;
    bool timed = false;
    bool prep_marked = false;
    bool scratch_dirty = true;          // counters / flags are not known to be zero (fresh slot or failed call)
    bool has_limbs = false;             // limbs / group scratch hold this call's rows (K3 can be re-run)
    int k3_images = 0, k3_first = 0;    // image range of the last K3 launch (single-range calls)
    CallCtx ctx = {};
    DevBuf<float> redo_lr, redo_hr;      // per-plane redo: fused network-resolution planes, their full-resolution maps
    DevBuf<int32_t> redo_list;
};

struct og_handle {
    og_config cfg;
    SkeletonDev sk;
    int device;
    int warp_rows;               // person-table rows of the one-warp-per-image K3 kernel (0 = off)
    int result_rows;             // pose rows per image the pinned result buffer starts with
    int64_t launches;

    // stand-alone stage APIs (og_nms_topk_f32, og_group_f32, ...): scratch in caller-stream order
    DevBuf<uint32_t> cand_count;
    DevBuf<uint64_t> cand_keys;
    GroupScratch group;
    cudaStream_t cp;                    // host API: input copies, one image range ahead of the kernels
    int sm_count;
    DevBuf<float> fused_hmp, fused_off;     // materialising path only
    DevBuf<float> hr_hmp, hr_off;
    FlipTablesDev ft;                   // flip-test tables, passed to the kernels by value
    uint64_t tables_version;

    ResultSlot slots[kSlots];
    int queue[kSlots];           // slots of the calls in flight, oldest first (ring buffer)
    int tail;                    // position of the oldest unfetched call in `queue`
    int pending;                 // decode calls in flight
    int last_slot;               // slot of the most recent decode call (intermediates)
    int fetched_slot;            // slot of the most recently fetched result (stage times)

    bool fused_enabled;
    bool graph_enabled;          // device path: replay a captured CUDA graph per slot
    bool zero_copy_enabled;      // host API: K2 gathers offsets straight from pinned host memory
    int64_t fused_redos;
    int64_t k3_redos;            // fetches that ran the CTA grouping kernel for images the warp kernel gave up
    int64_t zero_copy_calls;
    int64_t graph_replays, graph_builds;
    uint64_t graph_clock;
    bool tables_valid;           // ft matches the cached host copies
    int32_t kp_cache[OG_MAX_KEYPOINTS];
    int32_t limb_cache[OG_MAX_LIMBS];
    uint8_t reserved_cache[OG_MAX_LIMBS];

    bool timing;
    struct Plan {                // og_plan_features_strided: the arguments of a repeated device-path decode
        MapView hmp, off;        // validated at plan time
        int n, hgt, w, hmp_stride, off_stride, resize_mode, flip_test;
        uint64_t tables_version;
    };
    Plan *plans;
    int n_plans, cap_plans;
    double *staged_frames;       // og_set_frames: frames of the NEXT decode call
    int staged_n, staged_cap;
};

namespace {

// Result buffer of a slot: [meta][pose rows][result-row keypoints][result-row scores][result-row images]
inline size_t align16(size_t x) { return (x + 15) / 16 * 16; }
struct ResultLayout {
    size_t poses, coco_kp, coco_score, coco_image, total;
};
inline ResultLayout result_layout(const og_handle *h, int n, int capacity_rows) {
    const size_t c = (size_t)h->cfg.n_keypoints;
    ResultLayout lo;
    lo.poses = ((size_t)(2 * n + 2) * sizeof(int32_t) + 15) / 16 * 16;
    lo.coco_kp = align16(lo.poses + (size_t)capacity_rows * c * OG_POSE_COLS * sizeof(float));
    lo.coco_score = align16(lo.coco_kp + (size_t)capacity_rows * c * 3 * sizeof(float));
    lo.coco_image = align16(lo.coco_score + (size_t)capacity_rows * sizeof(double));
    lo.total = align16(lo.coco_image + (size_t)capacity_rows * sizeof(int32_t));
    return lo;
}

CocoOut coco_out(const og_handle *h, const ResultSlot *slot, int image0) {
    CocoOut c = {nullptr, nullptr, nullptr, nullptr, image0};
    if (!slot->emit_coco) return c;
    const ResultLayout lo = result_layout(h, slot->n, slot->capacity_rows);
    c.frames = slot->frames_dev;
    c.keypoints = reinterpret_cast<float *>(slot->out_dev + lo.coco_kp);
    c.scores = reinterpret_cast<double *>(slot->out_dev + lo.coco_score);
    c.images = reinterpret_cast<int32_t *>(slot->out_dev + lo.coco_image);
    return c;
}

// meta words: offset[n], count[n], overflow flag of the fused path, one spare
inline size_t meta_bytes_for(int n) { return ((size_t)(2 * n + 2) * sizeof(int32_t) + 15) / 16 * 16; }
int check_device(const og_handle *h) {
    int cur = -1;
    OG_CUDA_TRY(cudaGetDevice(&cur));
    OG_REQUIRE(cur == h->device, "handle is bound to CUDA device %d but the current device is %d",
               h->device, cur);
    return OG_OK;
}

int check_maps(int n, int hgt, int w, int c) {
    OG_REQUIRE(n >= 0 && hgt > 0 && w > 0, "bad map shape n=%d h=%d w=%d", n, hgt, w);
    OG_REQUIRE((long long)c * hgt * w < (1LL << 31), "C*H*W = %lld does not fit 31 bits",
               (long long)c * hgt * w);
    return OG_OK;
}

inline int mark(og_handle *h, ResultSlot *slot, int which, cudaStream_t s) {
    if (h->timing) OG_CUDA_TRY(cudaEventRecord(slot->ev[which], s));
    return OG_OK;
}

// ensure() that reports a moved buffer (a captured graph holds the old address)
template <typename Buf>
int ensure_tracked(Buf &buf, size_t need, ResultSlot *slot) {
    const auto *before = buf.ptr;
    OG_TRY(buf.ensure(need));
    if (buf.ptr != before) slot->buffers_version += 1;
    return OG_OK;
}

int ensure_result(og_handle *h, ResultSlot *slot, size_t bytes) {
    if (bytes <= slot->out_cap) return OG_OK;
    if (slot->out_host) OG_CUDA_TRY(cudaFreeHost(slot->out_host));
    slot->out_host = slot->out_dev = nullptr;
    slot->out_cap = 0;
    const size_t grow = bytes + bytes / 4;
    OG_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&slot->out_host), grow, cudaHostAllocMapped));
    OG_CUDA_TRY(cudaHostGetDevicePointer(reinterpret_cast<void **>(&slot->out_dev), slot->out_host, 0));
    slot->out_cap = grow;
    slot->buffers_version += 1;
    (void)h;
    return OG_OK;
}

// Slot of a new decode call; `forced` re-uses a slot (the redo of a fetched-but-overflowed batch).
int acquire_slot(og_handle *h, ResultSlot *forced, ResultSlot **out) {
    if (forced) {
        *out = forced;
        return OG_OK;
    }
    // the lowest free slot: a caller that keeps d calls in flight touches d slots (a synchronous
    // caller one), so only those ever allocate their buffers and capture graphs
    OG_REQUIRE(h->pending < kSlots,
               "%d decode calls are already in flight; call og_fetch_result before the next decode", kSlots);
    for (int i = 0; i < kSlots; ++i)
        if (!h->slots[i].pending) {
            *out = &h->slots[i];
            return OG_OK;
        }
    set_error("internal: no free result slot");
    return OG_ERR_CAPACITY;
}

int run_k1(og_handle *h, const float *heat, int n, int hgt, int w, float thre, float *score,
           int32_t *index, int32_t *count, cudaStream_t s, cudaEvent_t after_pass1 = nullptr) {
    const int planes = n * h->cfg.n_keypoints;
    OG_TRY(h->cand_count.ensure(planes));
    OG_TRY(h->cand_keys.ensure((size_t)planes * kCandCap));
    return launch_nms_topk(heat, planes, hgt, w, thre, h->cfg.topk, h->cand_count.ptr,
                           h->cand_keys.ptr, score, index, count, false, true, s, &h->launches,
                           after_pass1);
}

GroupLaunch group_launch(const og_handle *h, int n) {
    const og_config &c = h->cfg;
    GroupLaunch g = {};
    g.n = n;
    g.c = c.n_keypoints;
    g.l = c.n_limbs;
    g.k = c.topk;
    g.sk = h->sk;
    g.dist_max = c.dist_max;
    g.use_scale = c.use_scale;
    g.person_thre = c.person_thre;
    g.sort_dim = c.sort_dim;
    g.warp_rows = h->warp_rows;
    return g;
}

// Buffers K2's prepare tail and K3 need for n images.
int ensure_group_scratch(og_handle *h, GroupScratch &gs, int n, ResultSlot *slot) {
    GroupLaunch g = group_launch(h, n);
    const og_config &c = h->cfg;
    const size_t slab = ((size_t)c.n_limbs * c.topk * c.n_keypoints * 6 + 3) / 4 * 4 * (size_t)n;
    if (slot) {
        OG_TRY(ensure_tracked(gs.prep, group_prep_ints(g), slot));
        OG_TRY(ensure_tracked(gs.rec, group_rec_vec4(g), slot));
        OG_TRY(ensure_tracked(gs.cnt, (size_t)n * c.n_limbs, slot));
        OG_TRY(ensure_tracked(gs.redo, (size_t)n, slot));
        OG_TRY(ensure_tracked(gs.slab, slab, slot));
    } else {
        OG_TRY(gs.prep.ensure(group_prep_ints(g)));
        OG_TRY(gs.rec.ensure(group_rec_vec4(g)));
        OG_TRY(gs.cnt.ensure((size_t)n * c.n_limbs));
        OG_TRY(gs.redo.ensure((size_t)n));
        OG_TRY(gs.slab.ensure(slab));
    }
    return OG_OK;
}

// K3 on `n` images whose scratch rows start at image `i0` of the scratch buffers.
int run_k3(og_handle *h, GroupScratch &gs, int i0, const float *limbs, bool prepared, int n,
           float *out_poses, int capacity_rows, int32_t *out_offset, int32_t *out_count,
           int32_t *out_total, cudaStream_t s, const CocoOut *coco = nullptr, int32_t *lazy_flag = nullptr,
           bool redo_only = false) {
    const og_config &c = h->cfg;
    GroupLaunch g = group_launch(h, n);
    if (coco) g.coco = *coco;
    g.lazy_flag = lazy_flag;
    g.prep = gs.prep.ptr + (size_t)i0 * c.n_limbs * (c.topk + 1);
    g.rec = gs.rec.ptr + (size_t)i0 * c.n_limbs * c.topk * 3;
    g.cnt = gs.cnt.ptr + (size_t)i0 * c.n_limbs;
    g.redo = gs.redo.ptr + i0;
    g.slab_stride = ((size_t)c.n_limbs * c.topk * c.n_keypoints * 6 + 3) / 4 * 4;
    g.slab = gs.slab.ptr + (size_t)i0 * g.slab_stride;
    if (redo_only)
        return launch_group_redo(g, limbs, out_poses, capacity_rows, out_offset, out_count, out_total, s,
                                 &h->launches);
    return launch_group(g, limbs, prepared, out_poses, capacity_rows, out_offset, out_count, out_total, s,
                        &h->launches);
}

inline MapView dense_f32(const float *p, size_t per_image, size_t hw) {
    return MapView::planar(p, OG_DTYPE_F32, per_image, hw);
}
inline size_t elem_size(int dtype) { return dtype == OG_DTYPE_F32 ? 4 : 2; }
inline MapView shift_images(MapView v, size_t images) {
    v.ptr = static_cast<const char *>(v.ptr) + images * v.image_stride * elem_size(v.dtype);
    return v;
}

// One decode call = begin_call, decode_range over one or more image ranges, finish_call.
// begin_call: buffers of the slot (nothing is allocated after this point: the ranges may be
// captured into a graph), counters known to be zero, first stage mark.
int begin_call(og_handle *h, ResultSlot *slot, const K1Fused *fused, int n, int hgt, int w, cudaStream_t s) {
    const og_config &c = h->cfg;
    OG_TRY(check_maps(n, hgt, w, c.n_keypoints));
    const size_t dets = (size_t)n * c.n_keypoints * c.topk;
    OG_TRY(ensure_tracked(slot->det_score, dets, slot));
    OG_TRY(ensure_tracked(slot->det_index, dets, slot));
    OG_TRY(ensure_tracked(slot->det_count, (size_t)n * c.n_keypoints, slot));
    OG_TRY(ensure_tracked(slot->limbs, (size_t)n * c.n_limbs * c.topk * OG_LIMB_COLS, slot));
    OG_TRY(ensure_tracked(slot->total, 4, slot));
    // Pose rows: every person consumes at least one limb row, so n * L * K rows can never
    // overflow; real scenes hold tens of persons per image, so the pinned buffer starts at 64
    // rows per image and og_fetch_poses re-runs K3 into a worst-case buffer if a batch ever
    // needs more (it sees the counts either way).
    const long long worst = (long long)n * c.n_limbs * c.topk;
    int capacity_rows = (int)std::min<long long>(worst, std::max<long long>((long long)n * h->result_rows, 256));
    if (h->result_rows < 64) capacity_rows = (int)std::min<long long>(worst, (long long)n * h->result_rows);   // test aid
    const size_t mbytes = meta_bytes_for(n);
    if (slot->out_cap >= result_layout(h, n, (int)worst).total) capacity_rows = (int)worst;
    OG_TRY(ensure_result(h, slot, result_layout(h, n, capacity_rows).total));
    // image frames staged by og_set_frames belong to this call
    slot->emit_coco = false;
    if (h->staged_n >= 0) {
        const int staged = h->staged_n;
        h->staged_n = -1;
        OG_REQUIRE(staged == n, "og_set_frames staged %d image frames but the decode call has %d images", staged, n);
        if (n > slot->frames_cap) {
            if (slot->frames_host) OG_CUDA_TRY(cudaFreeHost(slot->frames_host));
            slot->frames_host = slot->frames_dev = nullptr;
            slot->frames_cap = 0;
            const int grow = n + n / 4 + 8;
            OG_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&slot->frames_host), (size_t)grow * 4 * sizeof(double),
                                      cudaHostAllocMapped));
            OG_CUDA_TRY(cudaHostGetDevicePointer(reinterpret_cast<void **>(&slot->frames_dev), slot->frames_host, 0));
            slot->frames_cap = grow;
            slot->buffers_version += 1;
        }
        memcpy(slot->frames_host, h->staged_frames, (size_t)n * 4 * sizeof(double));
        slot->emit_coco = n > 0;
    }
    const int planes = n * c.n_keypoints;
    bool fresh_scratch = slot->scratch_dirty;
    if (n > 0) {
        const uint32_t *before = slot->cand_count.ptr;
        OG_TRY(ensure_tracked(slot->cand_count, planes, slot));
        fresh_scratch = fresh_scratch || slot->cand_count.ptr != before;
        OG_TRY(ensure_tracked(slot->cand_keys, (size_t)planes * kCandCap, slot));
        OG_TRY(ensure_group_scratch(h, slot->group, n, slot));
        if (fused) {
            size_t flag_bytes = 0, tiles = 0;
            fused_scratch(n, c.n_keypoints, fused->h, fused->w, fused->scale, &flag_bytes, &tiles);
            const uint8_t *fb = slot->tile_flag.ptr;
            const int32_t *lb = slot->tile_list.ptr;
            OG_TRY(ensure_tracked(slot->tile_flag, flag_bytes, slot));
            OG_TRY(ensure_tracked(slot->tile_list, tiles + 4, slot));
            fresh_scratch = fresh_scratch || slot->tile_flag.ptr != fb || slot->tile_list.ptr != lb;
            if (fused->hmp.is_channels_last())
                OG_TRY(ensure_tracked(slot->nhwc_heat, (size_t)n * c.n_keypoints * fused->h * fused->w, slot));
        }
    }
    if (fresh_scratch) {
        // the kernels keep these zero from call to call; a new buffer (or a failed call) does not
        cudaStream_t w = slot->work;
        if (slot->cand_count.ptr) OG_CUDA_TRY(cudaMemsetAsync(slot->cand_count.ptr, 0, slot->cand_count.cap * sizeof(uint32_t), w));
        if (slot->tile_flag.ptr) OG_CUDA_TRY(cudaMemsetAsync(slot->tile_flag.ptr, 0, slot->tile_flag.cap, w));
        if (slot->tile_list.ptr) OG_CUDA_TRY(cudaMemsetAsync(slot->tile_list.ptr, 0, slot->tile_list.cap * sizeof(int32_t), w));
        OG_CUDA_TRY(cudaMemsetAsync(slot->total.ptr, 0, 4 * sizeof(int32_t), w));
        OG_CUDA_TRY(cudaStreamSynchronize(w));
    }
    slot->scratch_dirty = true;            // until finish_call: an error in between leaves them unknown
    slot->n = n;
    slot->meta_bytes = mbytes;
    slot->capacity_rows = capacity_rows;
    slot->stream = s;
    slot->fused = fused != nullptr;
    slot->timed = false;
    slot->has_limbs = false;
    if (!slot->prep_marked) OG_TRY(mark(h, slot, 0, s));
    slot->prep_marked = false;
    if (n > 0) {
        reinterpret_cast<volatile int32_t *>(slot->out_host)[2 * n] = 0;          // candidate-list overflow flag
        reinterpret_cast<volatile int32_t *>(slot->out_host)[2 * n + 1] = 0;      // K3: images left to the CTA kernel
    }
    return OG_OK;
}

// K2 (+ the row preparation of K3) and K3 of images [i0, i0 + cn) on the slot's stream; the dets of
// those images are in the slot's det arrays.
int run_limbs_and_groups(og_handle *h, ResultSlot *slot, int chunk, int i0, int cn, const float *offs,
                         const OffsetSource *offs_lowres, const FlipTablesDev *ft, const float *scales,
                         int hgt, int w, const LimbExtras *extras, bool timed) {
    const og_config &c = h->cfg;
    const int n = slot->n;
    int32_t *meta = reinterpret_cast<int32_t *>(slot->out_dev);
    float *poses = reinterpret_cast<float *>(slot->out_dev + slot->meta_bytes);
    const size_t HW = (size_t)hgt * w;
    const size_t det0 = (size_t)i0 * c.n_keypoints * c.topk;
    const size_t plane0 = (size_t)i0 * c.n_keypoints;
    const float *det_score = slot->det_score.ptr + det0;
    const int32_t *det_index = slot->det_index.ptr + det0;
    cudaStream_t a = slot->work;
    if (timed) OG_TRY(mark(h, slot, 4, a));
    const int nd = extras ? extras->vector_nd : 2;
    OffsetSource src = {};
    if (offs_lowres) {
        src = *offs_lowres;
        src.maps = shift_images(src.maps, i0);
    }
    LimbExtras ex = {nullptr, 2, 0};
    if (extras) {
        ex = *extras;
        if (ex.jomps) ex.jomps += (size_t)i0 * 2 * HW;
    }
    float *limbs = slot->limbs.ptr + (size_t)i0 * c.n_limbs * c.topk * OG_LIMB_COLS;
    GroupScratch &gs = slot->group;
    PrepOut po = {gs.prep.ptr + (size_t)i0 * c.n_limbs * (c.topk + 1),
                  gs.rec.ptr + (size_t)i0 * c.n_limbs * c.topk * 3, gs.cnt.ptr + (size_t)i0 * c.n_limbs,
                  c.dist_max, c.use_scale, chunk == 0 ? slot->total.ptr : nullptr};
    OG_TRY(launch_limb_score(det_score, det_index, offs ? offs + (size_t)i0 * nd * c.n_limbs * HW : nullptr,
                             offs_lowres ? &src : nullptr, ft, scales ? scales + plane0 * HW : nullptr,
                             extras ? &ex : nullptr, cn, c.n_keypoints, c.n_limbs, c.topk, hgt, w, h->sk,
                             c.thre_hmp, c.min_len, c.resize_factor, limbs, &po, a));
    h->launches += 1;
    if (timed) OG_TRY(mark(h, slot, 5, a));
    const CocoOut coco = coco_out(h, slot, i0);
    // A call that is one range leaves the images whose person table outgrows the warp kernel's
    // (noise-like inputs) to og_fetch_result: the kernel raises meta[2n + 1] and the fetch runs the
    // CTA kernel for them, instead of a launch of early-exit CTAs behind every call.
    int32_t *lazy_flag = (i0 == 0 && cn == n) ? meta + 2 * n + 1 : nullptr;
    OG_TRY(run_k3(h, gs, i0, limbs, true, cn, poses, slot->capacity_rows, meta + i0, meta + n + i0,
                  slot->total.ptr, a, &coco, lazy_flag));
    if (timed) OG_TRY(mark(h, slot, 6, a));
    slot->k3_first = i0;
    slot->k3_images = cn;
    return OG_OK;
}

// Images [i0, i0 + cn) of the call.  K1 (full-resolution stream, or the fused network-resolution
// kernels) on `k1s`, then K2 -> K3 on the slot's stream `a`; when both are the same stream the
// whole range is one linear chain (device path; this is what gets captured into a graph) and
// the kernels clear each other's counters instead of memsets.  `timed` ranges record the stage
// events (the last range of a call).  All map pointers address image 0 of the call.
int decode_range(og_handle *h, ResultSlot *slot, int chunk, int i0, int cn, const float *heat,
                 const K1Fused *fused, const float *offs, const OffsetSource *offs_lowres,
                 const float *scales, int hgt, int w, cudaStream_t k1s, const LimbExtras *extras,
                 bool timed) {
    const og_config &c = h->cfg;
    const int n = slot->n;
    int32_t *meta = reinterpret_cast<int32_t *>(slot->out_dev);
    const size_t HW = (size_t)hgt * w;
    const size_t det0 = (size_t)i0 * c.n_keypoints * c.topk;
    const size_t plane0 = (size_t)i0 * c.n_keypoints;
    float *det_score = slot->det_score.ptr + det0;
    int32_t *det_index = slot->det_index.ptr + det0;
    int32_t *det_count = slot->det_count.ptr + plane0;
    uint32_t *cand_count = slot->cand_count.ptr + plane0;
    uint64_t *cand_keys = slot->cand_keys.ptr + plane0 * kCandCap;
    const int planes = cn * c.n_keypoints;
    cudaStream_t a = slot->work;
    const bool chain = k1s == a;
    if (timed) OG_TRY(mark(h, slot, 1, k1s));
    int32_t *n_active = nullptr;
    if (fused) {
        n_active = slot->tile_list.ptr;
        // the mirrored copy of image i sits n images behind it: shifting the base keeps that offset
        OG_TRY(launch_fused_candidates(shift_images(fused->hmp, i0), h->ft, cn, n,
                                       c.n_keypoints, fused->h, fused->w, fused->scale, fused->cubic,
                                       fused->flip, c.thre_hmp, cand_count, cand_keys, slot->tile_flag.ptr,
                                       slot->tile_list.ptr + 4, n_active,
                                       slot->nhwc_heat.ptr ? slot->nhwc_heat.ptr + plane0 * fused->h * fused->w : nullptr,
                                       h->sm_count, !chain, k1s, &h->launches));
    } else {
        OG_TRY(launch_nms_candidates(heat + plane0 * HW, planes, hgt, w, c.thre_hmp, cand_count, cand_keys,
                                     k1s, &h->launches));
    }
    if (timed) OG_TRY(mark(h, slot, 2, k1s));
    // Host / full-resolution paths: everything after the streaming pass runs on the slot's own
    // high-priority stream — the per-plane selection, K2 and K3 are latency-bound and occupy
    // a fraction of the SMs, so the next K1 pass (HBM-bound, on the caller's stream) overlaps
    // them instead of queueing behind them.
    // On the full-resolution path the per-plane selection stays on the caller's stream: on the
    // slot's stream it slows the next streaming pass down (profiles/r1_stream_sweep.txt).
    const bool sel_on_aux = chain || fused != nullptr;
    if (!chain && sel_on_aux) {
        OG_CUDA_TRY(cudaEventRecord(slot->k1_done[chunk], k1s));
        OG_CUDA_TRY(cudaStreamWaitEvent(a, slot->k1_done[chunk], 0));
    }
    cudaStream_t sel = sel_on_aux ? a : k1s;
    if (timed) OG_TRY(mark(h, slot, 3, sel));
    OG_TRY(launch_select_topk(fused ? nullptr : heat + plane0 * HW, planes, hgt, w, c.thre_hmp, c.topk,
                              cand_count, cand_keys, det_score, det_index, det_count,
                              fused ? meta + 2 * n : nullptr,
                              // the active-block counter must be zero when the next call on this slot
                              // starts: the chain's selection clears it, and so does the selection of
                              // the LAST range of a host call (earlier ranges clear it with a memset
                              // before their scan, because the next range's scan may already run)
                              (chain || timed) ? n_active : nullptr, sel));
    h->launches += 1;
    if (!chain && !sel_on_aux) {
        OG_CUDA_TRY(cudaEventRecord(slot->k1_done[chunk], k1s));
        OG_CUDA_TRY(cudaStreamWaitEvent(a, slot->k1_done[chunk], 0));
    }
    if (fused && offs_lowres) {
        slot->ctx = CallCtx{*fused, *offs_lowres, h->ft, hgt, w, LimbExtras{}};
        if (extras) slot->ctx.extras = *extras;
    }
    return run_limbs_and_groups(h, slot, chunk, i0, cn, offs, offs_lowres, &h->ft, scales, hgt, w, extras, timed);
}

int finish_call(og_handle *h, ResultSlot *slot) {
    const int n = slot->n;
    if (n > 0) {
        cudaStream_t a = slot->work;
        OG_TRY(mark(h, slot, 7, a));
        slot->timed = h->timing;
        OG_CUDA_TRY(cudaEventRecord(slot->done, a));
        slot->has_limbs = true;
    }
    slot->scratch_dirty = false;
    if (!slot->pending) {           // a redo keeps its place in the queue
        slot->pending = true;
        h->queue[(h->tail + h->pending) % kSlots] = (int)(slot - h->slots);
        h->pending += 1;
    }
    h->last_slot = (int)(slot - h->slots);
    return OG_OK;
}

// The whole batch as one range (full-resolution maps, or the materialising features path):
// K1 on the caller's stream, the rest on the slot's.
int decode_core(og_handle *h, ResultSlot *slot, const float *heat, const K1Fused *fused,
                const float *offs, const OffsetSource *offs_lowres, const float *scales, int n,
                int hgt, int w, cudaStream_t s, const LimbExtras *extras = nullptr) {
    OG_TRY(begin_call(h, slot, fused, n, hgt, w, s));
    if (n > 0)
        OG_TRY(decode_range(h, slot, 0, 0, n, heat, fused, offs, offs_lowres, scales, hgt, w, s, extras, true));
    else
        OG_TRY(mark(h, slot, 1, s));
    return finish_call(h, slot);
}

// Device path of the fused decode: the caller's stream is only waited on; the whole chain
// (K1f scan -> list -> blocks -> select -> K2 + prepare -> K3) runs on the slot's stream, so
// calls in flight overlap each other and the caller's stream is free at once.  Without stage
// timing the chain is a CUDA graph captured once per slot and replayed while the inputs, the
// shapes and the slot's buffers stay the same: one cudaGraphLaunch instead of six kernel
// launches.
int decode_chain(og_handle *h, ResultSlot *slot, const K1Fused &k1, const OffsetSource &src, int n,
                 int H, int W, cudaStream_t s, const LimbExtras *extras = nullptr) {
    OG_TRY(begin_call(h, slot, &k1, n, H, W, s));
    cudaStream_t a = slot->work;
    if (n == 0) {
        OG_TRY(mark(h, slot, 1, s));
        return finish_call(h, slot);
    }
    OG_CUDA_TRY(cudaEventRecord(slot->call_start, s));
    OG_CUDA_TRY(cudaStreamWaitEvent(a, slot->call_start, 0));
    // what this call runs on, for a redo at fetch time (a graph replay does not pass through
    // decode_range, and the slot may have served other buffers since the graph was captured)
    slot->ctx = CallCtx{k1, src, h->ft, H, W, LimbExtras{}};
    if (extras) slot->ctx.extras = *extras;
    if (!h->graph_enabled || h->timing) {
        OG_TRY(decode_range(h, slot, 0, 0, n, nullptr, &k1, nullptr, &src, nullptr, H, W, a, extras, true));
        return finish_call(h, slot);
    }
    const GraphKey key = {k1.hmp.ptr, src.maps.ptr, k1.hmp.dtype, k1.hmp.image_stride, src.maps.image_stride,
                          k1.hmp.plane_stride, k1.hmp.pixel_stride, src.maps.plane_stride, src.maps.pixel_stride,
                          n, k1.h, k1.w, k1.scale, k1.cubic ? 1 : 0, k1.flip ? 1 : 0, slot->emit_coco ? 1 : 0,
                          h->tables_version, slot->buffers_version,
                          extras ? extras->scale_lr.maps : MapView(), extras ? extras->jitter_lr.maps : MapView(),
                          extras ? extras->vector_nd : 2, extras ? extras->use_jitter : 0};
    int gi = -1, victim = 0;
    for (int i = 0; i < kGraphsPerSlot; ++i) {
        if (slot->graph[i] != nullptr && slot->key[i] == key) gi = i;
        if (slot->graph_used[i] < slot->graph_used[victim]) victim = i;
    }
    if (gi < 0) {
        gi = victim;
        cudaGraph_t graph = nullptr;
        OG_CUDA_TRY(cudaStreamBeginCapture(a, cudaStreamCaptureModeRelaxed));
        const int st = decode_range(h, slot, 0, 0, n, nullptr, &k1, nullptr, &src, nullptr, H, W, a, extras, false);
        const cudaError_t end = cudaStreamEndCapture(a, &graph);
        if (st != OG_OK) {
            if (graph) cudaGraphDestroy(graph);
            return st;
        }
        OG_CUDA_TRY(end);
        bool updated = false;
        if (slot->graph[gi] != nullptr) {
            cudaGraphExecUpdateResultInfo info;
            updated = cudaGraphExecUpdate(slot->graph[gi], graph, &info) == cudaSuccess;
            if (!updated) {
                (void)cudaGetLastError();
                cudaGraphExecDestroy(slot->graph[gi]);
                slot->graph[gi] = nullptr;
            }
        }
        if (!updated) {
            const cudaError_t inst = cudaGraphInstantiate(&slot->graph[gi], graph, 0);
            if (inst != cudaSuccess) {
                cudaGraphDestroy(graph);
                slot->graph[gi] = nullptr;
                OG_CUDA_TRY(inst);
            }
        }
        cudaGraphDestroy(graph);
        slot->key[gi] = key;
        h->graph_builds += 1;
    } else {
        h->launches += 6;           // scan, list, blocks, select, K2, K3: the graph's kernel nodes
        slot->k3_first = 0;
        slot->k3_images = n;
    }
    slot->graph_used[gi] = ++h->graph_clock;
    OG_CUDA_TRY(cudaGraphLaunch(slot->graph[gi], a));
    h->graph_replays += 1;
    return finish_call(h, slot);
}

int upload_flip_tables(og_handle *h, const int32_t *kp_flip, const int32_t *limb_flip,
                       const int32_t *limb_reserve, int n_reserve) {
    const og_config &c = h->cfg;
    OG_REQUIRE(kp_flip && limb_flip && (n_reserve == 0 || limb_reserve),
               "flip_test needs the keypoint / limb flip tables");
    uint8_t reserved[OG_MAX_LIMBS] = {0};
    for (int i = 0; i < c.n_keypoints; ++i)
        OG_REQUIRE(kp_flip[i] >= 0 && kp_flip[i] < c.n_keypoints, "kp_flip[%d] out of range", i);
    for (int i = 0; i < c.n_limbs; ++i)
        OG_REQUIRE(limb_flip[i] >= 0 && limb_flip[i] < c.n_limbs, "limb_flip[%d] out of range", i);
    for (int i = 0; i < n_reserve; ++i) {
        OG_REQUIRE(limb_reserve[i] >= 0 && limb_reserve[i] < c.n_limbs, "limb_reserve[%d] out of range", i);
        reserved[limb_reserve[i]] = 1;
    }
    if (h->tables_valid && memcmp(h->kp_cache, kp_flip, sizeof(int32_t) * c.n_keypoints) == 0 &&
        memcmp(h->limb_cache, limb_flip, sizeof(int32_t) * c.n_limbs) == 0 &&
        memcmp(h->reserved_cache, reserved, c.n_limbs) == 0)
        return OG_OK;                      // unchanged
    // the tables travel by value with every launch: nothing on the device to update or wait for
    memset(&h->ft, 0, sizeof(h->ft));
    for (int i = 0; i < c.n_keypoints; ++i) h->ft.kp[i] = (int8_t)kp_flip[i];
    for (int i = 0; i < c.n_limbs; ++i) {
        h->ft.limb[i] = (int8_t)limb_flip[i];
        if (reserved[i]) h->ft.reserved |= 1ull << i;
    }
    memcpy(h->kp_cache, kp_flip, sizeof(int32_t) * c.n_keypoints);
    memcpy(h->limb_cache, limb_flip, sizeof(int32_t) * c.n_limbs);
    memcpy(h->reserved_cache, reserved, c.n_limbs);
    h->tables_valid = true;
    h->tables_version += 1;
    return OG_OK;
}

int decode_features_impl(og_handle *h, ResultSlot *slot, const float *hmp, const float *off, int n,
                         int hgt, int w, int hmp_stride, int off_stride, int resize_mode,
                         int flip_test, cudaStream_t s, bool allow_fused) {
    const og_config &c = h->cfg;
    const float *cur_h = hmp, *cur_o = off;
    const size_t hw = (size_t)hgt * w;
    if (!slot->prep_marked) {
        OG_TRY(mark(h, slot, 0, s));
        slot->prep_marked = h->timing;
    }

    // Fused path: candidates straight from the network-resolution maps, offsets sampled at
    // the candidates; no full-resolution map is written.  thre_hmp <= 0 (every pixel is a
    // candidate) and other strides use the materialising path below.
    if (allow_fused && h->fused_enabled && c.thre_hmp > 0.0f &&
        fused_supported(n, c.n_keypoints, hmp_stride, hgt, w)) {
        OG_TRY(check_maps(n, hgt * hmp_stride, w * hmp_stride, c.n_keypoints));
        K1Fused k1 = {dense_f32(hmp, (size_t)c.n_keypoints * hw, hw), hgt, w, hmp_stride, resize_mode == 1,
                      flip_test != 0};
        OffsetSource src = {dense_f32(off, (size_t)2 * c.n_limbs * hw, hw), hgt, w, off_stride,
                            flip_test ? 1 : 0, n};
        return decode_chain(h, slot, k1, src, n, hgt * hmp_stride, w * hmp_stride, s);
    }
    // Materialising path: the flip / resize outputs below are handle-owned and still read by
    // K2 of an earlier call on its slot's stream, so this call's writes wait for those calls.
    for (int i = 0; i < kSlots; ++i)
        if (&h->slots[i] != slot && h->slots[i].pending && h->slots[i].n > 0)
            OG_CUDA_TRY(cudaStreamWaitEvent(s, h->slots[i].done, 0));
    if (flip_test) {
        OG_TRY(h->fused_hmp.ensure((size_t)n * c.n_keypoints * hw));
        OG_TRY(h->fused_off.ensure((size_t)n * 2 * c.n_limbs * hw));
        OG_TRY(launch_flip_fuse(cur_h, cur_o, h->ft, n, c.n_keypoints, c.n_limbs, hgt, w, h->fused_hmp.ptr,
                                h->fused_off.ptr, s));
        h->launches += 1;
        cur_h = h->fused_hmp.ptr;
        cur_o = h->fused_off.ptr;
    }
    int H = hgt, W = w;
    if (hmp_stride > 1) {
        H = hgt * hmp_stride;
        W = w * hmp_stride;
        OG_TRY(check_maps(n, H, W, c.n_keypoints));
        OG_TRY(h->hr_hmp.ensure((size_t)n * c.n_keypoints * H * W));
        OG_TRY(h->hr_off.ensure((size_t)n * 2 * c.n_limbs * H * W));
        OG_TRY(launch_resize(cur_h, h->hr_hmp.ptr, n * c.n_keypoints, hgt, w, hmp_stride, resize_mode, s));
        OG_TRY(launch_resize(cur_o, h->hr_off.ptr, n * 2 * c.n_limbs, hgt, w, off_stride, 0, s));
        h->launches += 2;
        cur_h = h->hr_hmp.ptr;
        cur_o = h->hr_off.ptr;
    }
    return decode_core(h, slot, cur_h, nullptr, cur_o, nullptr, nullptr, n, H, W, s);
}

// The frames staged by og_set_frames belong to the next decode call, whether that call runs or is
// refused: one on every og_decode_* entry point drops them on return, so that a refused call does
// not hand its frames to the call after it (begin_call has taken them over when the call runs).
struct StagedFramesOfCall {
    og_handle *h;
    ~StagedFramesOfCall() {
        if (h) h->staged_n = -1;
    }
};

int check_feature_args(og_handle *h, int n, int hgt, int w, int hmp_stride, int off_stride,
                       int resize_mode, int flip_test, const int32_t *kp_flip,
                       const int32_t *limb_flip, const int32_t *limb_reserve, int n_reserve) {
    OG_TRY(check_device(h));
    OG_TRY(check_maps(n, hgt, w, h->cfg.n_keypoints));
    OG_REQUIRE(hmp_stride >= 1 && off_stride >= 1, "strides must be >= 1");
    OG_REQUIRE(hmp_stride == off_stride,
               "heat and offset maps must reach the same resolution (collect.py:81): strides %d vs %d",
               hmp_stride, off_stride);
    OG_REQUIRE(resize_mode == 0 || resize_mode == 1, "resize_mode must be 0 (bilinear) or 1 (bicubic)");
    if (flip_test) OG_TRY(upload_flip_tables(h, kp_flip, limb_flip, limb_reserve, n_reserve));
    return OG_OK;
}

}  // namespace

extern "C" {

const char *og_last_error(void) { return og::g_error; }

const char *og_status_string(int status) {
    switch (status) {
        case OG_OK: return "ok";
        case OG_ERR_INVALID_ARGUMENT: return "invalid argument";
        case OG_ERR_CUDA: return "CUDA error";
        case OG_ERR_OUT_OF_MEMORY: return "out of memory";
        case OG_ERR_CAPACITY: return "output capacity exceeded";
        case OG_ERR_UNSUPPORTED: return "unsupported configuration";
        default: return "unknown status";
    }
}

int og_abi_version(void) { return OG_ABI_VERSION; }

int og_create(const og_config *cfg, og_handle **out) {
    OG_REQUIRE(cfg && out, "og_create: null argument");
    *out = nullptr;
    OG_REQUIRE(cfg->n_keypoints >= 1 && cfg->n_keypoints <= OG_MAX_KEYPOINTS,
               "n_keypoints %d outside [1, %d]", cfg->n_keypoints, OG_MAX_KEYPOINTS);
    OG_REQUIRE(cfg->n_limbs >= 1 && cfg->n_limbs <= OG_MAX_LIMBS, "n_limbs %d outside [1, %d]",
               cfg->n_limbs, OG_MAX_LIMBS);
    OG_REQUIRE(cfg->topk >= 1 && cfg->topk <= OG_MAX_TOPK, "topk %d outside [1, %d]", cfg->topk,
               OG_MAX_TOPK);
    OG_REQUIRE(cfg->limb_from && cfg->limb_to, "skeleton tables missing");
    OG_REQUIRE(cfg->sort_dim >= 0 && cfg->sort_dim < OG_POSE_COLS, "sort_dim %d outside [0, 6)",
               cfg->sort_dim);
    OG_REQUIRE((long long)cfg->n_limbs * cfg->topk < 32768, "n_limbs * topk must stay below 32768");
    for (int i = 0; i < cfg->n_limbs; ++i) {
        OG_REQUIRE(cfg->limb_from[i] >= 0 && cfg->limb_from[i] < cfg->n_keypoints &&
                       cfg->limb_to[i] >= 0 && cfg->limb_to[i] < cfg->n_keypoints,
                   "limb %d references a keypoint outside [0, %d)", i, cfg->n_keypoints);
    }
    int device = cfg->device;
    if (device < 0) {
        OG_CUDA_TRY(cudaGetDevice(&device));
    } else {
        int cur = -1;
        OG_CUDA_TRY(cudaGetDevice(&cur));
        OG_REQUIRE(cur == device, "og_create: make device %d current first (current is %d)", device, cur);
    }
    cudaDeviceProp prop;
    OG_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("this library is built for sm_100a (B200); device %d is sm_%d%d", device, prop.major,
                  prop.minor);
        return OG_ERR_UNSUPPORTED;
    }

    og_handle *h = new (std::nothrow) og_handle();
    if (!h) {
        set_error("host allocation failed");
        return OG_ERR_OUT_OF_MEMORY;
    }
    h->cfg = *cfg;
    h->cfg.limb_from = nullptr;
    h->cfg.limb_to = nullptr;
    for (int i = 0; i < cfg->n_limbs; ++i) {
        h->sk.from[i] = cfg->limb_from[i];
        h->sk.to[i] = cfg->limb_to[i];
    }
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    h->launches = 0;
    h->tail = h->pending = 0;
    h->last_slot = 0;
    h->fetched_slot = -1;
    h->timing = false;
    h->cp = nullptr;
    h->fused_enabled = true;
    h->graph_enabled = true;
    h->graph_replays = h->graph_builds = 0;
    h->k3_redos = 0;
    h->graph_clock = 0;
    h->plans = nullptr;
    h->n_plans = h->cap_plans = 0;
    h->staged_frames = nullptr;
    h->staged_n = -1;
    h->staged_cap = 0;
    h->result_rows = 64;
    if (const char *env = getenv("OG_RESULT_ROWS")) {          // test aid: force the regroup path
        const int v = atoi(env);
        if (v >= 1) h->result_rows = v;
    }
    h->tables_version = 1;
    memset(&h->ft, 0, sizeof(h->ft));
    h->zero_copy_enabled = true;
    h->fused_redos = 0;
    h->zero_copy_calls = 0;
    h->tables_valid = false;

    // Supported sizes: the CTA grouping kernel's shared work arrays for L * K persons plus a margin
    // of 16 person rows (C * 24 bytes each) fit in 200 KB.  The kernel does not need the margin; it
    // keeps the limit where the tests reach (the 64-keypoint ring at K = 96 is the largest such
    // configuration), and a larger limit needs tests at the new sizes.
    GroupLaunch g = {};
    g.c = cfg->n_keypoints;
    g.l = cfg->n_limbs;
    g.k = cfg->topk;
    const int pmax = cfg->n_limbs * cfg->topk;
    const size_t group_smem = group_smem_bytes(g);
    const size_t supported = std::min<size_t>(prop.sharedMemPerBlockOptin, 200 * 1024);
    if (group_smem + (size_t)16 * cfg->n_keypoints * 24 > supported) {
        delete h;
        set_error("n_limbs * topk = %d needs %zu bytes of shared work arrays; unsupported", pmax, group_smem);
        return OG_ERR_UNSUPPORTED;
    }
    // One-warp-per-image kernel: 64 person rows (26 KB of shared memory for 17 keypoints, eight
    // images per SM) hold every real scene; an image that needs more is redone by the CTA kernel.
    h->warp_rows = std::min(64, pmax);
    if (const char *env = getenv("OG_K3_WARP_ROWS")) {         // test aid; 0 = CTA kernel only
        const int v = atoi(env);
        if (v >= 0 && v <= 256) h->warp_rows = std::min(v, pmax);
    }
    g.warp_rows = h->warp_rows;
    while (g.warp_rows > 8 && group_warp_smem_bytes(g) > 96 * 1024) g.warp_rows /= 2;
    h->warp_rows = g.warp_rows;
    int st = prepare_group_kernel(group_smem, group_warp_smem_bytes(g));
    if (st != OG_OK) {
        delete h;
        return st;
    }
    {
        int least = 0, greatest = 0;
        cudaError_t err = cudaDeviceGetStreamPriorityRange(&least, &greatest);
        for (int i = 0; i < kSlots && err == cudaSuccess; ++i)
            err = cudaStreamCreateWithPriority(&h->slots[i].work, cudaStreamNonBlocking, greatest);
        if (err != cudaSuccess) {
            og_destroy(h);
            set_error("cudaStreamCreateWithPriority failed: %s", cudaGetErrorString(err));
            return OG_ERR_CUDA;
        }
    }
    if (cudaStreamCreateWithFlags(&h->cp, cudaStreamNonBlocking) != cudaSuccess) {
        h->cp = nullptr;
        og_destroy(h);
        set_error("cudaStreamCreateWithFlags failed");
        return OG_ERR_CUDA;
    }
    for (int i = 0; i < kSlots; ++i) {
        cudaError_t err = cudaEventCreateWithFlags(&h->slots[i].done, cudaEventDisableTiming);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&h->slots[i].call_start, cudaEventDisableTiming);
        for (int j = 0; j < kMaxChunks && err == cudaSuccess; ++j) {
            err = cudaEventCreateWithFlags(&h->slots[i].k1_done[j], cudaEventDisableTiming);
            if (err == cudaSuccess) err = cudaEventCreateWithFlags(&h->slots[i].copied[j], cudaEventDisableTiming);
        }
        if (err != cudaSuccess) {
            og_destroy(h);
            set_error("cudaEventCreate failed: %s", cudaGetErrorString(err));
            return OG_ERR_CUDA;
        }
    }
    *out = h;
    return OG_OK;
}

int og_destroy(og_handle *h) {
    if (!h) return OG_OK;
    cudaDeviceSynchronize();
    h->cand_count.release();
    h->cand_keys.release();
    h->group.release();
    h->fused_hmp.release();
    h->fused_off.release();
    h->hr_hmp.release();
    h->hr_off.release();
    for (int i = 0; i < kSlots; ++i) {
        ResultSlot &sl = h->slots[i];
        for (int g = 0; g < kGraphsPerSlot; ++g)
            if (sl.graph[g]) cudaGraphExecDestroy(sl.graph[g]);
        if (sl.out_host) cudaFreeHost(sl.out_host);
        if (sl.frames_host) cudaFreeHost(sl.frames_host);
        sl.total.release();
        sl.in_hmp.release();
        sl.in_off.release();
        sl.det_score.release();
        sl.det_index.release();
        sl.det_count.release();
        sl.cand_count.release();
        sl.cand_keys.release();
        sl.tile_flag.release();
        sl.tile_list.release();
        sl.nhwc_heat.release();
        sl.limbs.release();
        sl.redo_lr.release();
        sl.redo_hr.release();
        sl.redo_list.release();
        sl.group.release();
        if (sl.done) cudaEventDestroy(sl.done);
        if (sl.call_start) cudaEventDestroy(sl.call_start);
        for (int j = 0; j < kMaxChunks; ++j) {
            if (sl.k1_done[j]) cudaEventDestroy(sl.k1_done[j]);
            if (sl.copied[j]) cudaEventDestroy(sl.copied[j]);
        }
        for (int e = 0; e < kStageEvents; ++e)
            if (sl.ev[e]) cudaEventDestroy(sl.ev[e]);
        if (sl.work) cudaStreamDestroy(sl.work);
    }
    if (h->cp) cudaStreamDestroy(h->cp);
    free(h->staged_frames);
    free(h->plans);
    delete h;
    return OG_OK;
}

int og_hmp_nms_f32(const float *heat_dev, float *out_dev, int n, int c, int h, int w, void *stream) {
    OG_REQUIRE(heat_dev && out_dev, "og_hmp_nms_f32: null pointer");
    OG_TRY(check_maps(n, h, w, c));
    return launch_hmp_nms(heat_dev, out_dev, n * c, h, w, static_cast<cudaStream_t>(stream));
}

int og_topk_channel_f32(og_handle *h, const float *scores_dev, int n, int c, int hgt, int w, int k,
                        float *out_score_dev, int32_t *out_index_dev, void *stream) {
    OG_REQUIRE(h && scores_dev && out_score_dev && out_index_dev, "og_topk_channel_f32: null pointer");
    OG_TRY(check_device(h));
    OG_TRY(check_maps(n, hgt, w, c));
    OG_REQUIRE(k >= 1 && k <= kCandCap && (long long)k <= (long long)hgt * w,
               "k = %d outside [1, min(%d, H*W)]", k, kCandCap);
    return launch_nms_topk(scores_dev, n * c, hgt, w, -INFINITY, k, nullptr, nullptr, out_score_dev,
                           out_index_dev, nullptr, true, false, static_cast<cudaStream_t>(stream),
                           &h->launches);
}

int og_nms_topk_f32(og_handle *h, const float *heat_dev, int n, int hgt, int w, float thre,
                    float *out_score_dev, int32_t *out_index_dev, int32_t *out_count_dev,
                    void *stream) {
    OG_REQUIRE(h && heat_dev && out_score_dev && out_index_dev, "og_nms_topk_f32: null pointer");
    OG_TRY(check_device(h));
    OG_TRY(check_maps(n, hgt, w, h->cfg.n_keypoints));
    return run_k1(h, heat_dev, n, hgt, w, thre, out_score_dev, out_index_dev, out_count_dev,
                  static_cast<cudaStream_t>(stream));
}

int og_limb_score_f32(og_handle *h, const float *det_score_dev, const int32_t *det_index_dev,
                      const float *offs_dev, const float *scales_dev, int n, int hgt, int w,
                      float *out_limbs_dev, void *stream) {
    OG_REQUIRE(h && det_score_dev && det_index_dev && offs_dev && out_limbs_dev,
               "og_limb_score_f32: null pointer");
    OG_TRY(check_device(h));
    OG_TRY(check_maps(n, hgt, w, h->cfg.n_keypoints));
    const og_config &c = h->cfg;
    OG_TRY(launch_limb_score(det_score_dev, det_index_dev, offs_dev, nullptr, nullptr, scales_dev, nullptr, n,
                             c.n_keypoints, c.n_limbs, c.topk, hgt, w, h->sk, c.thre_hmp, c.min_len,
                             c.resize_factor, out_limbs_dev, nullptr, static_cast<cudaStream_t>(stream)));
    h->launches += 1;
    return OG_OK;
}

int og_limb_score_ex_f32(og_handle *h, const float *det_score_dev, const int32_t *det_index_dev,
                         const float *offs_dev, const float *scales_dev, const float *jomps_dev,
                         int vector_nd, int use_jitter, int n, int hgt, int w, float *out_limbs_dev,
                         void *stream) {
    OG_REQUIRE(h && det_score_dev && det_index_dev && offs_dev && out_limbs_dev,
               "og_limb_score_ex_f32: null pointer");
    OG_REQUIRE(vector_nd == 2 || vector_nd == 4, "vector_nd must be 2 or 4");
    OG_REQUIRE(!(vector_nd == 4 && jomps_dev && use_jitter),
               "jitter refinement of 4-D offset vectors is undefined (it raises in the reference too)");
    OG_TRY(check_device(h));
    OG_TRY(check_maps(n, hgt, w, h->cfg.n_keypoints));
    const og_config &c = h->cfg;
    LimbExtras ex = {jomps_dev, vector_nd, use_jitter};
    OG_TRY(launch_limb_score(det_score_dev, det_index_dev, offs_dev, nullptr, nullptr, scales_dev, &ex, n,
                             c.n_keypoints, c.n_limbs, c.topk, hgt, w, h->sk, c.thre_hmp, c.min_len,
                             c.resize_factor, out_limbs_dev, nullptr, static_cast<cudaStream_t>(stream)));
    h->launches += 1;
    return OG_OK;
}

int og_flip_average_f32(const float *in2n_dev, const int32_t *perm, int negate_even, int n, int ch,
                        int hgt, int w, float *out_dev, void *stream) {
    OG_REQUIRE(in2n_dev && out_dev, "og_flip_average_f32: null pointer");
    OG_REQUIRE(n >= 0 && ch >= 1 && ch <= 128 && hgt > 0 && w > 0, "og_flip_average_f32: bad shape");
    ChannelPerm p;
    for (int i = 0; i < ch; ++i) {
        p.src[i] = perm ? perm[i] : i;
        OG_REQUIRE(p.src[i] >= 0 && p.src[i] < ch, "og_flip_average_f32: perm[%d] out of range", i);
    }
    return launch_flip_average(in2n_dev, out_dev, n, ch, hgt, w, p, negate_even != 0,
                               static_cast<cudaStream_t>(stream));
}

int og_flip_cat_offsets_f32(const float *off2n_dev, const int32_t *limb_flip,
                            const int32_t *limb_reserve, int n_reserve, int n, int n_limbs, int hgt,
                            int w, float *out_dev, void *stream) {
    OG_REQUIRE(off2n_dev && out_dev && limb_flip, "og_flip_cat_offsets_f32: null pointer");
    OG_REQUIRE(n >= 0 && n_limbs >= 1 && n_limbs <= OG_MAX_LIMBS && hgt > 0 && w > 0,
               "og_flip_cat_offsets_f32: bad shape");
    ChannelPerm lf, rs;
    for (int i = 0; i < 128; ++i) rs.src[i] = 0;
    for (int i = 0; i < n_limbs; ++i) {
        lf.src[i] = limb_flip[i];
        OG_REQUIRE(lf.src[i] >= 0 && lf.src[i] < n_limbs, "limb_flip[%d] out of range", i);
    }
    for (int i = 0; i < n_reserve; ++i) {
        OG_REQUIRE(limb_reserve && limb_reserve[i] >= 0 && limb_reserve[i] < n_limbs,
                   "limb_reserve[%d] out of range", i);
        rs.src[limb_reserve[i]] = 1;
    }
    return launch_flip_cat_offsets(off2n_dev, out_dev, n, n_limbs, hgt, w, lf, rs,
                                   static_cast<cudaStream_t>(stream));
}

int og_group_f32(og_handle *h, const float *limbs_dev, int n, float *out_poses_dev,
                 int32_t capacity_rows, int32_t *out_offset_dev, int32_t *out_count_dev,
                 int32_t *out_total_dev, void *stream) {
    OG_REQUIRE(h && limbs_dev && out_poses_dev && out_offset_dev && out_count_dev && out_total_dev,
               "og_group_f32: null pointer");
    OG_REQUIRE(n >= 0 && capacity_rows >= 0, "og_group_f32: negative size");
    OG_TRY(check_device(h));
    if (n == 0) return OG_OK;
    // the stand-alone stage APIs share one scratch set, ordered by the caller's stream
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    OG_TRY(ensure_group_scratch(h, h->group, n, nullptr));
    OG_CUDA_TRY(cudaMemsetAsync(out_total_dev, 0, sizeof(int32_t), s));
    return run_k3(h, h->group, 0, limbs_dev, false, n, out_poses_dev, capacity_rows, out_offset_dev,
                  out_count_dev, out_total_dev, s);
}

int og_scored_offset_f32(og_handle *h, const float *hmp_dev, const float *off_dev, int n, int hgt,
                         int w, int kernel_size, float *out_dev, void *stream) {
    OG_REQUIRE(h && hmp_dev && off_dev && out_dev, "og_scored_offset_f32: null pointer");
    OG_REQUIRE(kernel_size >= 1 && (kernel_size & 1), "kernel_size must be odd and positive");
    OG_TRY(check_device(h));
    OG_TRY(check_maps(n, hgt, w, h->cfg.n_keypoints));
    OG_TRY(launch_scored_offset(hmp_dev, off_dev, n, h->cfg.n_keypoints, h->cfg.n_limbs, hgt, w,
                                kernel_size, h->sk, out_dev, static_cast<cudaStream_t>(stream)));
    h->launches += 1;
    return OG_OK;
}

int og_flip_fuse_f32(og_handle *h, const float *hmp2n_dev, const float *off2n_dev,
                     const int32_t *kp_flip, const int32_t *limb_flip, const int32_t *limb_reserve,
                     int n_reserve, int n, int hgt, int w, float *out_hmp_dev, float *out_off_dev,
                     void *stream) {
    OG_REQUIRE(h && hmp2n_dev && off2n_dev && out_hmp_dev && out_off_dev, "og_flip_fuse_f32: null pointer");
    OG_TRY(check_device(h));
    OG_TRY(check_maps(n, hgt, w, h->cfg.n_keypoints));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    OG_TRY(upload_flip_tables(h, kp_flip, limb_flip, limb_reserve, n_reserve));
    OG_TRY(launch_flip_fuse(hmp2n_dev, off2n_dev, h->ft, n, h->cfg.n_keypoints, h->cfg.n_limbs, hgt, w,
                            out_hmp_dev, out_off_dev, s));
    h->launches += 1;
    return OG_OK;
}

int og_resize_f32(const float *in_dev, float *out_dev, int planes, int hgt, int w, int scale,
                  int mode, void *stream) {
    OG_REQUIRE(in_dev && out_dev, "og_resize_f32: null pointer");
    OG_REQUIRE(planes >= 0 && hgt > 0 && w > 0 && scale >= 1, "og_resize_f32: bad shape");
    OG_REQUIRE(mode == 0 || mode == 1, "og_resize_f32: mode must be 0 (bilinear) or 1 (bicubic)");
    return launch_resize(in_dev, out_dev, planes, hgt, w, scale, mode, static_cast<cudaStream_t>(stream));
}

int og_decode_maps(og_handle *h, const float *heat_dev, const float *offs_dev,
                   const float *scales_dev, int n, int hgt, int w, void *stream) {
    StagedFramesOfCall frames_of_call{h};
    OG_REQUIRE(h && (n == 0 || (heat_dev && offs_dev)), "og_decode_maps: null pointer");
    OG_TRY(check_device(h));
    ResultSlot *slot = nullptr;
    OG_TRY(acquire_slot(h, nullptr, &slot));
    return decode_core(h, slot, heat_dev, nullptr, offs_dev, nullptr, scales_dev, n, hgt, w,
                       static_cast<cudaStream_t>(stream));
}

int og_decode_maps_ex(og_handle *h, const float *heat_dev, const float *offs_dev,
                      const float *scales_dev, const float *jomps_dev, int vector_nd, int use_jitter,
                      int n, int hgt, int w, void *stream) {
    StagedFramesOfCall frames_of_call{h};
    OG_REQUIRE(h && (n == 0 || (heat_dev && offs_dev)), "og_decode_maps_ex: null pointer");
    OG_REQUIRE(vector_nd == 2 || vector_nd == 4, "vector_nd must be 2 or 4");
    OG_REQUIRE(!(vector_nd == 4 && jomps_dev && use_jitter),
               "jitter refinement of 4-D offset vectors is undefined (it raises in the reference too)");
    OG_TRY(check_device(h));
    ResultSlot *slot = nullptr;
    OG_TRY(acquire_slot(h, nullptr, &slot));
    LimbExtras ex = {jomps_dev, vector_nd, use_jitter};
    return decode_core(h, slot, heat_dev, nullptr, offs_dev, nullptr, scales_dev, n, hgt, w,
                       static_cast<cudaStream_t>(stream), &ex);
}

int og_decode_features_dev(og_handle *h, const float *hmp_dev, const float *off_dev, int n, int hgt,
                           int w, int hmp_stride, int off_stride, int resize_mode, int flip_test,
                           const int32_t *kp_flip, const int32_t *limb_flip,
                           const int32_t *limb_reserve, int n_reserve, void *stream) {
    StagedFramesOfCall frames_of_call{h};
    OG_REQUIRE(h && (n == 0 || (hmp_dev && off_dev)), "og_decode_features_dev: null pointer");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    OG_TRY(check_feature_args(h, n, hgt, w, hmp_stride, off_stride, resize_mode, flip_test, kp_flip,
                              limb_flip, limb_reserve, n_reserve));
    ResultSlot *slot = nullptr;
    OG_TRY(acquire_slot(h, nullptr, &slot));
    return decode_features_impl(h, slot, hmp_dev, off_dev, n, hgt, w, hmp_stride, off_stride,
                                resize_mode, flip_test, s, true);
}

namespace {

// The view of one map from its element strides in (image, channel, row, column) order: planar
// (s_n, h * w, w, 1) or channels-last (s_n, 1, w * p, p) with p >= channels; s_n must cover an image
// unless the buffer holds a single one.  A layout that is both is planar.  Anything else is refused
// here, before any launch.
int map_view(const char *name, const void *ptr, int dtype, const int64_t st[4], int channels, int images, int hgt,
             int w, MapView *out) {
    OG_REQUIRE(st != nullptr, "%s: null stride array", name);
    const int64_t hw = (int64_t)hgt * w;
    if (st[3] == 1 && st[2] == w && st[1] == hw) {
        OG_REQUIRE(images <= 1 || st[0] >= channels * hw,
                   "%s: image stride %lld is smaller than one planar image (%lld elements)", name,
                   (long long)st[0], (long long)(channels * hw));
        *out = MapView::planar(ptr, dtype, (size_t)std::max<int64_t>(st[0], channels * hw), (size_t)hw);
        return OG_OK;
    }
    const int64_t p = st[3];
    OG_REQUIRE(st[1] == 1 && p >= channels && st[2] == w * p,
               "%s: strides (%lld, %lld, %lld, %lld) are neither planar (s_n, %lld, %d, 1) nor channels-last "
               "(s_n, 1, %d * p, p) with p >= %d channels", name, (long long)st[0], (long long)st[1],
               (long long)st[2], (long long)st[3], (long long)hw, w, w, channels);
    OG_REQUIRE(images <= 1 || st[0] >= hw * p,
               "%s: image stride %lld is smaller than one channels-last image (%lld elements)", name,
               (long long)st[0], (long long)(hw * p));
    *out = MapView::channels_last(ptr, dtype, (size_t)std::max<int64_t>(st[0], hw * p), (size_t)p);
    return OG_OK;
}

// og_decode_features_dev_strided / og_decode_features_heads_dev_strided behind their argument checks
// (also the body of a plan launch); `extras`: the optional heads and flags, which only the fused
// path decodes
int decode_dev_views(og_handle *h, const MapView &hv, const MapView &ov, int n, int hgt, int w, int hmp_stride,
                     int off_stride, int resize_mode, int flip_test, cudaStream_t s,
                     const LimbExtras *extras = nullptr) {
    const og_config &c = h->cfg;
    const size_t hw = (size_t)hgt * w;
    const size_t hmp_img = (size_t)c.n_keypoints * hw, off_img = (size_t)2 * c.n_limbs * hw;
    if (!extras && hv.dtype == OG_DTYPE_F32 && !hv.is_channels_last() && !ov.is_channels_last() &&
        hv.image_stride == hmp_img && ov.image_stride == off_img) {
        ResultSlot *slot = nullptr;
        OG_TRY(acquire_slot(h, nullptr, &slot));
        return decode_features_impl(h, slot, static_cast<const float *>(hv.ptr), static_cast<const float *>(ov.ptr),
                                    n, hgt, w, hmp_stride, off_stride, resize_mode, flip_test, s, true);
    }
    if (!(h->fused_enabled && c.thre_hmp > 0.0f && fused_supported(n, c.n_keypoints, hmp_stride, hgt, w))) {
        if (extras)
            set_error("og_decode_features_heads_dev needs the fused path (stride 2, 4 or 8, thre_hmp > 0, fused "
                      "enabled); resize the maps and call og_decode_maps_ex");
        else
            set_error("og_decode_features_dev_ex: bf16 / strided maps need the fused path (stride 2, 4 or 8, "
                      "thre_hmp > 0, fused enabled); convert to dense float32 and call og_decode_features_dev");
        return OG_ERR_UNSUPPORTED;
    }
    ResultSlot *slot = nullptr;
    OG_TRY(acquire_slot(h, nullptr, &slot));
    const int H = hgt * hmp_stride, W = w * hmp_stride;
    OG_TRY(check_maps(n, H, W, c.n_keypoints));
    K1Fused k1 = {hv, hgt, w, hmp_stride, resize_mode == 1, flip_test != 0};
    OffsetSource src = {ov, hgt, w, off_stride, flip_test ? 1 : 0, n};
    return decode_chain(h, slot, k1, src, n, H, W, s, extras);
}

int check_dtype(int dtype) {
    OG_REQUIRE(dtype == OG_DTYPE_F32 || dtype == OG_DTYPE_BF16 || dtype == OG_DTYPE_F16,
               "dtype must be OG_DTYPE_F32, OG_DTYPE_BF16 or OG_DTYPE_F16");
    return OG_OK;
}

// the element strides of og_decode_features_dev_ex's planar views (image stride 0 = dense)
int planar_strides(const char *name, int64_t image_stride, int channels, int hgt, int w, int64_t out[4]) {
    const int64_t hw = (int64_t)hgt * w;
    OG_REQUIRE(image_stride == 0 || image_stride >= channels * hw,
               "%s %lld is smaller than one image (%lld elements)", name, (long long)image_stride,
               (long long)(channels * hw));
    out[0] = image_stride ? image_stride : channels * hw;
    out[1] = hw;
    out[2] = w;
    out[3] = 1;
    return OG_OK;
}

// validated views of both maps
int feature_views(og_handle *h, const void *hmp_dev, const void *off_dev, int dtype, const int64_t *hmp_st,
                  const int64_t *off_st, int n, int hgt, int w, int flip_test, MapView *hv, MapView *ov) {
    const int images = flip_test ? 2 * n : n;
    OG_TRY(map_view("hmp_elem_strides", hmp_dev, dtype, hmp_st, h->cfg.n_keypoints, images, hgt, w, hv));
    OG_TRY(map_view("off_elem_strides", off_dev, dtype, off_st, 2 * h->cfg.n_limbs, images, hgt, w, ov));
    return OG_OK;
}

}  // namespace

int og_decode_features_dev_strided(og_handle *h, const void *hmp_dev, const void *off_dev, int dtype,
                                   const int64_t hmp_elem_strides[4], const int64_t off_elem_strides[4], int n,
                                   int hgt, int w, int hmp_stride, int off_stride, int resize_mode, int flip_test,
                                   const int32_t *kp_flip, const int32_t *limb_flip,
                                   const int32_t *limb_reserve, int n_reserve, void *stream) {
    StagedFramesOfCall frames_of_call{h};
    OG_REQUIRE(h && (n == 0 || (hmp_dev && off_dev)), "og_decode_features_dev_strided: null pointer");
    OG_TRY(check_dtype(dtype));
    OG_TRY(check_feature_args(h, n, hgt, w, hmp_stride, off_stride, resize_mode, flip_test, kp_flip,
                              limb_flip, limb_reserve, n_reserve));
    MapView hv, ov;
    OG_TRY(feature_views(h, hmp_dev, off_dev, dtype, hmp_elem_strides, off_elem_strides, n, hgt, w, flip_test, &hv,
                         &ov));
    return decode_dev_views(h, hv, ov, n, hgt, w, hmp_stride, off_stride, resize_mode, flip_test,
                            static_cast<cudaStream_t>(stream));
}

int og_decode_features_dev_ex(og_handle *h, const void *hmp_dev, const void *off_dev, int dtype,
                              int64_t hmp_image_stride, int64_t off_image_stride, int n, int hgt,
                              int w, int hmp_stride, int off_stride, int resize_mode, int flip_test,
                              const int32_t *kp_flip, const int32_t *limb_flip,
                              const int32_t *limb_reserve, int n_reserve, void *stream) {
    StagedFramesOfCall frames_of_call{h};
    OG_REQUIRE(h && (n == 0 || (hmp_dev && off_dev)), "og_decode_features_dev_ex: null pointer");
    OG_TRY(check_dtype(dtype));
    OG_TRY(check_feature_args(h, n, hgt, w, hmp_stride, off_stride, resize_mode, flip_test, kp_flip,
                              limb_flip, limb_reserve, n_reserve));
    int64_t hs[4], os[4];
    OG_TRY(planar_strides("hmp_image_stride", hmp_image_stride, h->cfg.n_keypoints, hgt, w, hs));
    OG_TRY(planar_strides("off_image_stride", off_image_stride, 2 * h->cfg.n_limbs, hgt, w, os));
    return og_decode_features_dev_strided(h, hmp_dev, off_dev, dtype, hs, os, n, hgt, w, hmp_stride, off_stride,
                                          resize_mode, flip_test, kp_flip, limb_flip, limb_reserve, n_reserve,
                                          stream);
}

int og_decode_features_heads_dev_strided(og_handle *h, const void *hmp_dev, const void *off_dev, const void *scale_dev,
                                         const void *jitter_dev, int dtype, const int64_t hmp_elem_strides[4],
                                         const int64_t off_elem_strides[4], const int64_t scale_elem_strides[4],
                                         const int64_t jitter_elem_strides[4], int n, int hgt, int w, int hmp_stride,
                                         int off_stride, int resize_mode, int flip_test, int cat_flip_offs,
                                         int use_jitter, const int32_t *kp_flip, const int32_t *limb_flip,
                                         const int32_t *limb_reserve, int n_reserve, void *stream) {
    StagedFramesOfCall frames_of_call{h};
    OG_REQUIRE(h && (n == 0 || (hmp_dev && off_dev)), "og_decode_features_heads_dev: null pointer");
    OG_REQUIRE(!cat_flip_offs || flip_test, "cat_flip_offs concatenates the mirrored copy's offsets: it needs flip_test");
    OG_REQUIRE(!(cat_flip_offs && jitter_dev && use_jitter),
               "jitter refinement of 4-D offset vectors is undefined (it raises in the reference too)");
    OG_TRY(check_dtype(dtype));
    OG_TRY(check_feature_args(h, n, hgt, w, hmp_stride, off_stride, resize_mode, flip_test, kp_flip,
                              limb_flip, limb_reserve, n_reserve));
    MapView hv, ov, sv, jv;
    OG_TRY(feature_views(h, hmp_dev, off_dev, dtype, hmp_elem_strides, off_elem_strides, n, hgt, w, flip_test, &hv,
                         &ov));
    const int images = flip_test ? 2 * n : n;
    if (scale_dev)
        OG_TRY(map_view("scale_elem_strides", scale_dev, dtype, scale_elem_strides, h->cfg.n_keypoints, images, hgt,
                        w, &sv));
    if (jitter_dev)
        OG_TRY(map_view("jitter_elem_strides", jitter_dev, dtype, jitter_elem_strides, 2, images, hgt, w, &jv));
    LimbExtras ex = {};
    ex.vector_nd = cat_flip_offs ? 4 : 2;
    ex.use_jitter = use_jitter ? 1 : 0;
    // keypoint scales are resized like the heat maps (x off_stride, inter_mode), jitter offsets
    // bilinearly x hmp_stride (factory.py:80-88)
    ex.scale_lr = HeadSource{sv, hgt, w, off_stride, resize_mode == 1 ? 1 : 0};
    ex.jitter_lr = HeadSource{jv, hgt, w, hmp_stride, 0};
    return decode_dev_views(h, hv, ov, n, hgt, w, hmp_stride, off_stride, resize_mode, flip_test,
                            static_cast<cudaStream_t>(stream), &ex);
}

int og_decode_features_heads_dev(og_handle *h, const float *hmp_dev, const float *off_dev,
                                 const float *scale_dev, const float *jitter_dev, int n, int hgt, int w,
                                 int hmp_stride, int off_stride, int resize_mode, int flip_test,
                                 int cat_flip_offs, int use_jitter, const int32_t *kp_flip,
                                 const int32_t *limb_flip, const int32_t *limb_reserve, int n_reserve,
                                 void *stream) {
    StagedFramesOfCall frames_of_call{h};
    OG_REQUIRE(h, "og_decode_features_heads_dev: null pointer");
    OG_TRY(check_maps(n, hgt, w, h->cfg.n_keypoints));
    int64_t hs[4], os[4], ss[4], js[4];
    OG_TRY(planar_strides("hmp", 0, h->cfg.n_keypoints, hgt, w, hs));
    OG_TRY(planar_strides("off", 0, 2 * h->cfg.n_limbs, hgt, w, os));
    OG_TRY(planar_strides("scale", 0, h->cfg.n_keypoints, hgt, w, ss));
    OG_TRY(planar_strides("jitter", 0, 2, hgt, w, js));
    return og_decode_features_heads_dev_strided(h, hmp_dev, off_dev, scale_dev, jitter_dev, OG_DTYPE_F32, hs, os,
                                                scale_dev ? ss : nullptr, jitter_dev ? js : nullptr, n, hgt, w,
                                                hmp_stride, off_stride, resize_mode, flip_test, cat_flip_offs,
                                                use_jitter, kp_flip, limb_flip, limb_reserve, n_reserve, stream);
}

int og_plan_features_strided(og_handle *h, const void *hmp_dev, const void *off_dev, int dtype,
                             const int64_t hmp_elem_strides[4], const int64_t off_elem_strides[4], int n, int hgt,
                             int w, int hmp_stride, int off_stride, int resize_mode, int flip_test,
                             const int32_t *kp_flip, const int32_t *limb_flip, const int32_t *limb_reserve,
                             int n_reserve, int32_t *plan_id) {
    OG_REQUIRE(h && plan_id, "og_plan_features: null pointer");
    *plan_id = -1;
    OG_TRY(check_feature_args(h, n, hgt, w, hmp_stride, off_stride, resize_mode, flip_test, kp_flip,
                              limb_flip, limb_reserve, n_reserve));
    if (h->n_plans == h->cap_plans) {
        const int cap = h->cap_plans ? 2 * h->cap_plans : 16;
        og_handle::Plan *grown = static_cast<og_handle::Plan *>(realloc(h->plans, (size_t)cap * sizeof(og_handle::Plan)));
        if (!grown) {
            set_error("host allocation failed");
            return OG_ERR_OUT_OF_MEMORY;
        }
        h->plans = grown;
        h->cap_plans = cap;
    }
    OG_REQUIRE(hmp_dev && off_dev && n > 0, "og_plan_features: null pointer or empty batch");
    OG_TRY(check_dtype(dtype));
    MapView hv, ov;
    OG_TRY(feature_views(h, hmp_dev, off_dev, dtype, hmp_elem_strides, off_elem_strides, n, hgt, w, flip_test, &hv,
                         &ov));
    h->plans[h->n_plans] = og_handle::Plan{hv, ov, n, hgt, w, hmp_stride, off_stride, resize_mode, flip_test,
                                           h->tables_version};
    *plan_id = h->n_plans++;
    return OG_OK;
}

int og_plan_features(og_handle *h, const void *hmp_dev, const void *off_dev, int dtype,
                     int64_t hmp_image_stride, int64_t off_image_stride, int n, int hgt, int w,
                     int hmp_stride, int off_stride, int resize_mode, int flip_test,
                     const int32_t *kp_flip, const int32_t *limb_flip, const int32_t *limb_reserve,
                     int n_reserve, int32_t *plan_id) {
    OG_REQUIRE(h && plan_id, "og_plan_features: null pointer");
    *plan_id = -1;
    OG_TRY(check_maps(n, hgt, w, h->cfg.n_keypoints));
    int64_t hs[4], os[4];
    OG_TRY(planar_strides("hmp_image_stride", hmp_image_stride, h->cfg.n_keypoints, hgt, w, hs));
    OG_TRY(planar_strides("off_image_stride", off_image_stride, 2 * h->cfg.n_limbs, hgt, w, os));
    return og_plan_features_strided(h, hmp_dev, off_dev, dtype, hs, os, n, hgt, w, hmp_stride, off_stride,
                                    resize_mode, flip_test, kp_flip, limb_flip, limb_reserve, n_reserve, plan_id);
}

int og_plan_launch(og_handle *h, int32_t plan_id, void *stream) {
    StagedFramesOfCall frames_of_call{h};
    OG_REQUIRE(h && plan_id >= 0 && plan_id < h->n_plans, "og_plan_launch: unknown plan %d", plan_id);
    const og_handle::Plan &p = h->plans[plan_id];
    OG_REQUIRE(!p.flip_test || p.tables_version == h->tables_version,
               "og_plan_launch: the flip tables changed since plan %d was made", plan_id);
    OG_TRY(check_device(h));
    return decode_dev_views(h, p.hmp, p.off, p.n, p.hgt, p.w, p.hmp_stride, p.off_stride, p.resize_mode,
                            p.flip_test, static_cast<cudaStream_t>(stream));
}

int og_decode_features_host(og_handle *h, const float *hmp_host, const float *off_host, int n,
                            int hgt, int w, int hmp_stride, int off_stride, int resize_mode,
                            int flip_test, const int32_t *kp_flip, const int32_t *limb_flip,
                            const int32_t *limb_reserve, int n_reserve, void *stream) {
    StagedFramesOfCall frames_of_call{h};
    OG_REQUIRE(h && (n == 0 || (hmp_host && off_host)), "og_decode_features_host: null pointer");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    OG_TRY(check_feature_args(h, n, hgt, w, hmp_stride, off_stride, resize_mode, flip_test, kp_flip,
                              limb_flip, limb_reserve, n_reserve));
    ResultSlot *slot = nullptr;
    OG_TRY(acquire_slot(h, nullptr, &slot));
    const og_config &c = h->cfg;
    const size_t n_in = (size_t)(flip_test ? 2 * n : n);
    const size_t hw = (size_t)hgt * w;
    const bool fuse = h->fused_enabled && c.thre_hmp > 0.0f &&
                      fused_supported(n, c.n_keypoints, hmp_stride, hgt, w);
    // Zero-copy offsets: on the fused path K2 reads 2 * L * K bilinear samples per image, a few
    // KB out of the 2L * h * w * 4 bytes of the offset maps.  When the caller's buffer is pinned
    // (device-accessible) host memory the maps are not copied at all; K2 gathers its samples over
    // PCIe.  Pageable buffers and the materialising path copy everything as before.
    const float *off_alias = nullptr;
    if (h->zero_copy_enabled && n_in && fuse) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, off_host) == cudaSuccess &&
            attr.type == cudaMemoryTypeHost && attr.devicePointer != nullptr)
            off_alias = static_cast<const float *>(attr.devicePointer);
        else
            (void)cudaGetLastError();       // not registered: clear the error state
    }
    const size_t hmp_img = (size_t)c.n_keypoints * hw, off_img = (size_t)2 * c.n_limbs * hw;
    OG_TRY(ensure_tracked(slot->in_hmp, std::max<size_t>(1, n_in * hmp_img), slot));
    if (!off_alias) OG_TRY(ensure_tracked(slot->in_off, std::max<size_t>(1, n_in * off_img), slot));
    OG_TRY(mark(h, slot, 0, s));
    slot->prep_marked = h->timing;

    // The copies run on the handle's copy stream, one image range ahead of the kernels: while
    // range j is decoded (K1f on `stream`, K2 / K3 on the slot's stream) range j + 1 crosses
    // PCIe.  The buffers are ready in `stream` order, so the copy stream starts behind it.
    OG_CUDA_TRY(cudaEventRecord(slot->call_start, s));
    OG_CUDA_TRY(cudaStreamWaitEvent(h->cp, slot->call_start, 0));
    // images [i0, i0 + cn) and, when flip-testing, their mirrored copies n images further on: one
    // 2-row strided copy (row pitch = n images) instead of two transfers
    auto copy_images = [&](float *dst, const float *src, size_t per_image, int i0, int cn) -> int {
        const size_t pitch = (size_t)n * per_image * sizeof(float), width = (size_t)cn * per_image * sizeof(float);
        if (flip_test && pitch <= 0x7fffffffULL) {          // within cudaMemcpy2D's pitch limit
            OG_CUDA_TRY(cudaMemcpy2DAsync(dst + (size_t)i0 * per_image, pitch, src + (size_t)i0 * per_image, pitch,
                                          width, 2, cudaMemcpyHostToDevice, h->cp));
            return OG_OK;
        }
        for (int half = 0; half < (flip_test ? 2 : 1); ++half) {
            const size_t at = ((size_t)half * n + i0) * per_image;
            OG_CUDA_TRY(cudaMemcpyAsync(dst + at, src + at, width, cudaMemcpyHostToDevice, h->cp));
        }
        return OG_OK;
    };
    auto copy_range = [&](int i0, int cn) -> int {
        OG_TRY(copy_images(slot->in_hmp.ptr, hmp_host, hmp_img, i0, cn));
        if (!off_alias) OG_TRY(copy_images(slot->in_off.ptr, off_host, off_img, i0, cn));
        return OG_OK;
    };
    const float *off_src = off_alias ? off_alias : slot->in_off.ptr;
    if (!fuse || n == 0) {                  // materialising path: one range
        if (n) OG_TRY(copy_range(0, n));
        OG_CUDA_TRY(cudaEventRecord(slot->copied[0], h->cp));
        OG_CUDA_TRY(cudaStreamWaitEvent(s, slot->copied[0], 0));
        return decode_features_impl(h, slot, slot->in_hmp.ptr, off_src, n, hgt, w, hmp_stride,
                                    off_stride, resize_mode, flip_test, s, false);
    }
    const int H = hgt * hmp_stride, W = w * hmp_stride;
    OG_TRY(check_maps(n, H, W, c.n_keypoints));
    K1Fused k1 = {dense_f32(slot->in_hmp.ptr, hmp_img, hw), hgt, w, hmp_stride, resize_mode == 1, flip_test != 0};
    OffsetSource src = {dense_f32(off_src, off_img, hw), hgt, w, off_stride, flip_test ? 1 : 0, n};
    OG_TRY(begin_call(h, slot, &k1, n, H, W, s));
    // Image ranges: only the kernels of the LAST range run after the last byte has arrived, so
    // that range is kept small (n / 16, at least 4 images); the others share the rest evenly.
    int bounds[kMaxChunks + 1];
    int ranges = 0;
    {
        const int tail = n >= 16 ? std::max(4, n / 16) : 0;
        const int body = n - tail, body_ranges = tail ? kMaxChunks - 1 : kMaxChunks;
        const int per = std::max((body + body_ranges - 1) / body_ranges, std::min(body, 4));
        bounds[0] = 0;
        for (int at = 0; at < body; at += per) bounds[++ranges] = std::min(at + per, body);
        if (tail) bounds[++ranges] = n;
    }
    for (int chunk = 0; chunk < ranges; ++chunk) {
        const int i0 = bounds[chunk], cn = bounds[chunk + 1] - i0;
        const bool last = chunk + 1 == ranges;
        OG_TRY(copy_range(i0, cn));
        OG_CUDA_TRY(cudaEventRecord(slot->copied[chunk], h->cp));
        OG_CUDA_TRY(cudaStreamWaitEvent(s, slot->copied[chunk], 0));
        OG_TRY(decode_range(h, slot, chunk, i0, cn, nullptr, &k1, nullptr, &src, nullptr, H, W, s, nullptr, last));
    }
    slot->k3_images = 0;                    // several K3 launches: a capacity redo regroups every range
    if (off_alias) h->zero_copy_calls += 1;
    return finish_call(h, slot);
}

namespace {

// Fused decode whose candidate lists overflowed in some planes (det_count == -1 there): each such
// plane is flip-fused at network resolution, resized to full resolution and selected by the exact
// radix selection, a group of planes per launch; then K2 / K3 of the whole call run again.
int redo_overflowed_planes(og_handle *h, ResultSlot *slot) {
    const og_config &c = h->cfg;
    const int n = slot->n, planes = n * c.n_keypoints;
    const CallCtx &ctx = slot->ctx;
    cudaStream_t a = slot->work;
    std::vector<int32_t> counts((size_t)planes), list;
    OG_CUDA_TRY(cudaMemcpyAsync(counts.data(), slot->det_count.ptr, sizeof(int32_t) * planes, cudaMemcpyDeviceToHost, a));
    OG_CUDA_TRY(cudaStreamSynchronize(a));
    for (int p = 0; p < planes; ++p)
        if (counts[p] < 0) list.push_back(p);
    if (!list.empty()) {
        const size_t hw = (size_t)ctx.k1.h * ctx.k1.w, HW = (size_t)ctx.H * ctx.W;
        const size_t group = std::max<size_t>(1, std::min(list.size(), ((size_t)256 << 20) / (HW * sizeof(float))));
        OG_TRY(ensure_tracked(slot->redo_list, list.size(), slot));
        OG_TRY(ensure_tracked(slot->redo_lr, group * hw, slot));
        OG_TRY(ensure_tracked(slot->redo_hr, group * HW, slot));
        OG_CUDA_TRY(cudaMemcpyAsync(slot->redo_list.ptr, list.data(), sizeof(int32_t) * list.size(),
                                    cudaMemcpyHostToDevice, a));
        for (size_t g0 = 0; g0 < list.size(); g0 += group) {
            const int cnt = (int)std::min(group, list.size() - g0);
            OG_TRY(launch_fuse_planes(ctx.k1.hmp, ctx.ft, n, c.n_keypoints, ctx.k1.h, ctx.k1.w, ctx.k1.flip,
                                      slot->redo_list.ptr + g0, cnt, slot->redo_lr.ptr, a));
            OG_TRY(launch_resize(slot->redo_lr.ptr, slot->redo_hr.ptr, cnt, ctx.k1.h, ctx.k1.w, ctx.k1.scale,
                                 ctx.k1.cubic ? 1 : 0, a));
            h->launches += 2;
            OG_TRY(launch_nms_topk(slot->redo_hr.ptr, cnt, ctx.H, ctx.W, c.thre_hmp, c.topk, nullptr, nullptr,
                                   slot->det_score.ptr, slot->det_index.ptr, slot->det_count.ptr, true, true, a,
                                   &h->launches, nullptr, slot->redo_list.ptr + g0));
        }
    }
    volatile int32_t *meta = reinterpret_cast<volatile int32_t *>(slot->out_host);
    meta[2 * n] = 0;
    meta[2 * n + 1] = 0;
    OG_TRY(run_limbs_and_groups(h, slot, 0, 0, n, nullptr, &ctx.src, &ctx.ft, nullptr, ctx.H, ctx.W,
                                ctx.extras.vector_nd ? &ctx.extras : nullptr, false));
    OG_CUDA_TRY(cudaStreamSynchronize(a));       // `list` is read by the copy above until here
    return OG_OK;
}

// Re-run K3 of a fetched call into a worst-case result buffer (more persons than the pinned
// buffer was sized for: noise-like inputs only).
int regroup_with_full_capacity(og_handle *h, ResultSlot *slot) {
    const og_config &c = h->cfg;
    const int n = slot->n;
    const long long worst = (long long)n * c.n_limbs * c.topk;
    OG_TRY(ensure_result(h, slot, result_layout(h, n, (int)worst).total));
    slot->capacity_rows = (int)worst;
    int32_t *meta = reinterpret_cast<int32_t *>(slot->out_dev);
    float *poses = reinterpret_cast<float *>(slot->out_dev + slot->meta_bytes);
    cudaStream_t a = slot->work;
    OG_CUDA_TRY(cudaMemsetAsync(slot->total.ptr, 0, sizeof(int32_t), a));
    const CocoOut coco = coco_out(h, slot, 0);
    OG_TRY(run_k3(h, slot->group, 0, slot->limbs.ptr, true, n, poses, slot->capacity_rows, meta, meta + n,
                  slot->total.ptr, a, &coco));
    OG_CUDA_TRY(cudaStreamSynchronize(a));
    return OG_OK;
}

}  // namespace

int og_fetch_result(og_handle *h, og_result *out) {
    OG_REQUIRE(h && out, "og_fetch_result: null pointer");
    memset(out, 0, sizeof(*out));
    OG_REQUIRE(h->pending > 0, "og_fetch_result: no decode call is pending");
    OG_TRY(check_device(h));
    ResultSlot *slot = &h->slots[h->queue[h->tail]];
    const int n = slot->n;
    long long total = 0;
    if (n > 0) {
        OG_CUDA_TRY(cudaStreamSynchronize(slot->work));
        const volatile int32_t *meta = reinterpret_cast<const volatile int32_t *>(slot->out_host);
        if (slot->fused && meta[2 * n] != 0) {
            // Some plane produced more than kCandCap candidates (noise-like input).  The fused kernel
            // cannot re-scan a map it never materialised, so those planes — and only those — are
            // materialised now and selected exactly, and K2 / K3 run again on the completed dets.
            h->fused_redos += 1;
            OG_TRY(redo_overflowed_planes(h, slot));
            meta = reinterpret_cast<const volatile int32_t *>(slot->out_host);
        }
        if (meta[2 * n + 1] != 0) {
            // some image's person table outgrew the warp kernel's rows: the CTA kernel (global
            // slab tables) groups those images now, appending their rows behind the others
            h->k3_redos += 1;
            int32_t *meta_dev = reinterpret_cast<int32_t *>(slot->out_dev);
            const CocoOut coco = coco_out(h, slot, 0);
            OG_TRY(run_k3(h, slot->group, 0, slot->limbs.ptr, true, n, reinterpret_cast<float *>(slot->out_dev + slot->meta_bytes),
                          slot->capacity_rows, meta_dev, meta_dev + n, slot->total.ptr, slot->work, &coco, nullptr, true));
            OG_CUDA_TRY(cudaStreamSynchronize(slot->work));
            reinterpret_cast<volatile int32_t *>(slot->out_host)[2 * n + 1] = 0;
        }
        for (int i = 0; i < n; ++i) total += meta[n + i];
        if (total > slot->capacity_rows) {       // rare: more persons than the pinned buffer was sized for
            OG_TRY(regroup_with_full_capacity(h, slot));
            meta = reinterpret_cast<const volatile int32_t *>(slot->out_host);
            total = 0;
            for (int i = 0; i < n; ++i) total += meta[n + i];
            if (total > slot->capacity_rows) {
                set_error("internal: %lld pose rows exceed the worst-case capacity %d", total, slot->capacity_rows);
                return OG_ERR_CAPACITY;
            }
        }
        out->offsets = reinterpret_cast<const int32_t *>(slot->out_host);
        out->counts = out->offsets + n;
        out->poses = reinterpret_cast<const float *>(slot->out_host + slot->meta_bytes);
        if (slot->emit_coco) {
            const ResultLayout lo = result_layout(h, n, slot->capacity_rows);
            out->coco_keypoints = reinterpret_cast<const float *>(slot->out_host + lo.coco_kp);
            out->coco_scores = reinterpret_cast<const double *>(slot->out_host + lo.coco_score);
            out->coco_images = reinterpret_cast<const int32_t *>(slot->out_host + lo.coco_image);
        }
    }
    out->n_images = n;
    out->total_rows = (int32_t)total;
    out->n_keypoints = h->cfg.n_keypoints;
    // identifies the pinned buffer behind the pointers (a binding can cache its views by it)
    out->buffer_id = (int32_t)((slot - h->slots) | ((slot->buffers_version & 0x3ffffff) << 4));
    slot->pending = false;
    h->pending -= 1;
    h->fetched_slot = h->queue[h->tail];
    h->tail = (h->tail + 1) % kSlots;
    return OG_OK;
}

int og_fetch_poses(og_handle *h, const float **poses_host, const int32_t **offset_host,
                   const int32_t **count_host, int32_t *total_rows) {
    OG_REQUIRE(h && poses_host && offset_host && count_host && total_rows, "og_fetch_poses: null pointer");
    og_result r;
    *poses_host = nullptr;
    *offset_host = nullptr;
    *count_host = nullptr;
    *total_rows = 0;
    OG_TRY(og_fetch_result(h, &r));
    *poses_host = r.poses;
    *offset_host = r.offsets;
    *count_host = r.counts;
    *total_rows = r.total_rows;
    return OG_OK;
}

int og_pending(const og_handle *h) { return h ? h->pending : 0; }

int og_copy_intermediates(og_handle *h, int n, float *det_score_dev, int32_t *det_index_dev,
                          float *limbs_dev, void *stream) {
    OG_REQUIRE(h, "og_copy_intermediates: null handle");
    OG_REQUIRE(n >= 0 && n <= h->slots[h->last_slot].n,
               "og_copy_intermediates: n = %d but the last decode had %d images", n,
               h->slots[h->last_slot].n);
    OG_TRY(check_device(h));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const og_config &c = h->cfg;
    ResultSlot *slot = &h->slots[h->last_slot];
    if (slot->n > 0) OG_CUDA_TRY(cudaStreamWaitEvent(s, slot->done, 0));     // K2 ran on the handle's stream
    const size_t dets = (size_t)n * c.n_keypoints * c.topk;
    if (det_score_dev && dets)
        OG_CUDA_TRY(cudaMemcpyAsync(det_score_dev, slot->det_score.ptr, dets * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (det_index_dev && dets)
        OG_CUDA_TRY(cudaMemcpyAsync(det_index_dev, slot->det_index.ptr, dets * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
    const size_t lim = (size_t)n * c.n_limbs * c.topk * OG_LIMB_COLS;
    if (limbs_dev && lim)
        OG_CUDA_TRY(cudaMemcpyAsync(limbs_dev, slot->limbs.ptr, lim * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return OG_OK;
}

int64_t og_launch_count(const og_handle *h) { return h ? h->launches : 0; }

int og_set_fused(og_handle *h, int enable) {
    OG_REQUIRE(h, "og_set_fused: null handle");
    h->fused_enabled = enable != 0;
    return OG_OK;
}

int64_t og_fused_redo_count(const og_handle *h) { return h ? h->fused_redos : 0; }

int64_t og_k3_redo_count(const og_handle *h) { return h ? h->k3_redos : 0; }

int og_set_zero_copy(og_handle *h, int enable) {
    OG_REQUIRE(h, "og_set_zero_copy: null handle");
    h->zero_copy_enabled = enable != 0;
    return OG_OK;
}

int64_t og_zero_copy_count(const og_handle *h) { return h ? h->zero_copy_calls : 0; }

int og_set_frames(og_handle *h, const double *frames_host, int n) {
    OG_REQUIRE(h && n >= 0 && (n == 0 || frames_host), "og_set_frames: null pointer");
    for (int i = 0; i < n; ++i)
        OG_REQUIRE(frames_host[4 * i + 2] != 0.0 && frames_host[4 * i + 3] != 0.0,
                   "og_set_frames: image %d has a zero scale", i);
    if (n > h->staged_cap) {
        double *grown = static_cast<double *>(realloc(h->staged_frames, (size_t)(n + 8) * 4 * sizeof(double)));
        if (!grown) {
            set_error("host allocation failed");
            return OG_ERR_OUT_OF_MEMORY;
        }
        h->staged_frames = grown;
        h->staged_cap = n + 8;
    }
    if (n) memcpy(h->staged_frames, frames_host, (size_t)n * 4 * sizeof(double));
    h->staged_n = n;
    return OG_OK;
}

int og_set_graph(og_handle *h, int enable) {
    OG_REQUIRE(h, "og_set_graph: null handle");
    h->graph_enabled = enable != 0;
    return OG_OK;
}

int64_t og_graph_replay_count(const og_handle *h) { return h ? h->graph_replays : 0; }
int64_t og_graph_build_count(const og_handle *h) { return h ? h->graph_builds : 0; }

int og_debug_k3_profile(uint64_t *out16, int reset) {
    OG_REQUIRE(out16, "og_debug_k3_profile: null pointer");
    return read_k3_profile(reinterpret_cast<unsigned long long *>(out16), reset != 0);
}

int og_enable_stage_timing(og_handle *h, int enable) {
    OG_REQUIRE(h, "og_enable_stage_timing: null handle");
    OG_TRY(check_device(h));
    if (enable) {
        for (int i = 0; i < kSlots; ++i)
            for (int e = 0; e < kStageEvents; ++e)
                if (!h->slots[i].ev[e]) OG_CUDA_TRY(cudaEventCreate(&h->slots[i].ev[e]));
    }
    h->timing = enable != 0;
    return OG_OK;
}

int og_last_stage_times_ms(og_handle *h, float *out6) {
    OG_REQUIRE(h && out6, "og_last_stage_times_ms: null pointer");
    OG_REQUIRE(h->fetched_slot >= 0 && h->slots[h->fetched_slot].timed,
               "og_last_stage_times_ms: enable stage timing, decode and fetch first");
    ResultSlot *slot = &h->slots[h->fetched_slot];
    OG_CUDA_TRY(cudaEventSynchronize(slot->ev[kStageEvents - 1]));
    static const int first[6] = {0, 1, 3, 4, 5, 6};     // ev[2] -> ev[3] is the hand-over between streams
    for (int i = 0; i < 6; ++i)
        OG_CUDA_TRY(cudaEventElapsedTime(&out6[i], slot->ev[first[i]], slot->ev[first[i] + 1]));
    return OG_OK;
}

}  // extern "C"
