// Shared declarations of the sm_100a decoder library (internal; the public ABI is
// include/og_decoder.h).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/og_decoder.h"

namespace og {

// ---- error plumbing --------------------------------------------------------
void set_error(const char *fmt, ...);

#define OG_CUDA_TRY(expr)                                                          \
    do {                                                                           \
        cudaError_t err__ = (expr);                                                \
        if (err__ != cudaSuccess) {                                                \
            og::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr,       \
                          cudaGetErrorString(err__));                              \
            return err__ == cudaErrorMemoryAllocation ? OG_ERR_OUT_OF_MEMORY       \
                                                       : OG_ERR_CUDA;              \
        }                                                                          \
    } while (0)

#define OG_REQUIRE(cond, ...)                                                      \
    do {                                                                           \
        if (!(cond)) {                                                             \
            og::set_error(__VA_ARGS__);                                            \
            return OG_ERR_INVALID_ARGUMENT;                                        \
        }                                                                          \
    } while (0)

#define OG_TRY(expr)                                                               \
    do {                                                                           \
        int st__ = (expr);                                                         \
        if (st__ != OG_OK) return st__;                                            \
    } while (0)

// ---- one shared-memory carve-out for every kernel of the decode chains ------------------
// An SM changes its L1 / shared-memory split only when it is empty.  The chains of several calls
// are in flight at once, so kernels that need no shared memory (the HBM-streaming passes) share the
// SMs with kernels that need 3 .. 26 KB per CTA; left to the default ("the smallest split that
// fits this kernel") every such neighbour forces SMs to drain before its CTAs can start — measured
// on the full-resolution path: K1 0.266 -> 0.305 ms when the kernel running beside it grew from
// 2.5 to 10.5 KB of shared memory per CTA.  All chain kernels therefore ask for the same split.
constexpr int kChainCarveoutPercent = 58;      // -> 132 KB shared memory, 96 KB L1 per SM

#ifdef __CUDACC__
template <auto Kernel>
inline void prefer_chain_carveout() {
    static unsigned long long done = 0ull;      // one bit per device; a repeated call is harmless
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return;
    if ((done >> dev) & 1ull) return;
    if (cudaFuncSetAttribute(Kernel, cudaFuncAttributePreferredSharedMemoryCarveout, kChainCarveoutPercent) !=
        cudaSuccess)
        (void)cudaGetLastError();
    done |= 1ull << dev;
}
#endif

// ---- K1 candidate buffers --------------------------------------------------
// Survivors of "3x3 peak and value >= thre" are appended per (image, channel)
// plane as 64-bit keys: high word = ~ordered(value), low word = flat index, so an
// ascending key order is (value desc, index asc).
constexpr int kCandCap = 2048;        // per-plane capacity; overflow -> radix path

__device__ __forceinline__ uint32_t ordered_bits(float v) {
    uint32_t u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float from_ordered_bits(uint32_t o) {
    uint32_t u = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
    return __uint_as_float(u);
}
__device__ __forceinline__ uint64_t make_key(float v, uint32_t idx) {
    return ((uint64_t)(~ordered_bits(v)) << 32) | idx;
}
__device__ __forceinline__ float key_value(uint64_t key) {
    return from_ordered_bits(~(uint32_t)(key >> 32));
}

// ---- launchers (one per .cu file) -------------------------------------------
struct SkeletonDev {
    int32_t from[OG_MAX_LIMBS];
    int32_t to[OG_MAX_LIMBS];
};

int launch_hmp_nms(const float *heat, float *out, int planes, int h, int w, cudaStream_t s);

// pass 1: stream the heat map, append survivors; pass 2: per-plane select.
// `force_radix` skips pass 1 and runs the exact radix selection on every plane;
// `apply_nms` = 0 selects on the raw map (topK_channel).  `plane_map` (device, optional): the
// results of plane b go to slot plane_map[b] of the output arrays.
int launch_nms_topk(const float *heat, int planes, int h, int w, float thre, int k,
                    uint32_t *cand_count, uint64_t *cand_keys,
                    float *out_score, int32_t *out_index, int32_t *out_count,
                    bool force_radix, bool apply_nms, cudaStream_t s, int64_t *launches,
                    cudaEvent_t after_pass1 = nullptr, const int32_t *plane_map = nullptr);
// pass 1 alone (counters cleared, survivors appended)
int launch_nms_candidates(const float *heat, int planes, int h, int w, float thre,
                          uint32_t *cand_count, uint64_t *cand_keys, cudaStream_t s,
                          int64_t *launches);
// pass 2 alone on candidate lists some other kernel filled; with heat == nullptr a plane
// with more than kCandCap candidates cannot be re-scanned: it raises *overflow_flag and its
// out_count is -1 (og_fetch_result materialises and selects such planes one by one).
// Every plane's counter is left at ZERO for the next call (the lists are per result slot);
// `clear_word`, when given, is zeroed as well (the fused path's active-block counter).
int launch_select_topk(const float *heat, int planes, int h, int w, float thre, int k,
                       uint32_t *cand_count, const uint64_t *cand_keys, float *out_score,
                       int32_t *out_index, int32_t *out_count, int32_t *overflow_flag,
                       int32_t *clear_word, cudaStream_t s);

// ---- network-resolution maps as the caller holds them ------------------------------
// Element types: float32 (what the reference decodes, factory.py:59), or bfloat16 / float16
// straight from a reduced-precision head (SURVEY 8f-4).  Such a value widens exactly to float32, so everything after the
// load is the float32 path bit for bit.  Images may be `image_stride` elements apart (channel
// slices of one packed [N, 55, h, w] network output).  Cell (y, x) of channel ch of image i is
// element i * image_stride + ch * plane_stride + (y * w + x) * pixel_stride: planar maps have
// plane_stride = h * w, pixel_stride = 1; channels-last (NHWC) maps plane_stride = 1 and
// pixel_stride = the channel count of the whole packed tensor.  Built through the factories only,
// so no view can leave a stride unset.
struct MapView {
    const void *ptr = nullptr;
    int dtype = OG_DTYPE_F32;       // OG_DTYPE_F32 / OG_DTYPE_BF16 / OG_DTYPE_F16
    size_t image_stride = 0;        // elements between consecutive images
    size_t plane_stride = 0;        // elements between consecutive channels
    size_t pixel_stride = 1;        // elements between consecutive cells of a row
    MapView() = default;
    static MapView planar(const void *p, int dtype, size_t image_stride, size_t hw) {
        return MapView(p, dtype, image_stride, hw, 1);
    }
    static MapView channels_last(const void *p, int dtype, size_t image_stride, size_t pixel_stride) {
        return MapView(p, dtype, image_stride, 1, pixel_stride);
    }
    bool is_channels_last() const { return pixel_stride != 1; }

private:
    MapView(const void *p, int dt, size_t is, size_t ps, size_t xs)
        : ptr(p), dtype(dt), image_stride(is), plane_stride(ps), pixel_stride(xs) {}
};
#ifdef __CUDACC__
__device__ __forceinline__ float load_cell(const float *p) { return __ldg(p); }
__device__ __forceinline__ float load_cell(const __nv_bfloat16 *p) {
    return __uint_as_float((unsigned)__ldg(reinterpret_cast<const unsigned short *>(p)) << 16);
}
__device__ __forceinline__ float load_cell(const __half *p) {
    return __half2float(__ushort_as_half(__ldg(reinterpret_cast<const unsigned short *>(p))));
}
#endif

// Offsets still at network resolution (fused path): K2 samples them bilinearly at the
// candidate pixels instead of gathering from a materialised full-resolution map.
// Flip-test tables (config/coco_data.py:119-153), passed to the kernels BY VALUE: they live in
// the constant bank, so no kernel waits on a dependent global load for them and the handle keeps
// no device copies.
struct FlipTablesDev {
    int8_t kp[OG_MAX_KEYPOINTS];    // heat-map channel of the mirrored image that matches channel c
    int8_t limb[OG_MAX_LIMBS];      // limb type of the mirrored image that matches limb l
    uint64_t reserved;              // bit l: limb l is its own mirror image, keep the original offsets
};

struct OffsetSource {
    MapView maps;                   // [n or 2n][2L][h][w], planar or channels-last
    int h, w, scale;                // network resolution and the x scale to decode resolution
    int flip, n;                    // flip: maps = n originals then n mirrored copies
};

// An optional head at NETWORK resolution (float32, dense [n or 2n][channels][h][w]; the flip layout
// and image count are those of the OffsetSource of the call): K2 interpolates it at the few
// pixels it needs instead of reading a materialised x scale map.
struct HeadSource {
    const float *ptr;       // nullptr: head not present
    int h, w, scale;
    int cubic;              // interpolation of the reference's resize (factory.py:80-88)
};

// Optional variants of generate_limbs (collect.py:127-138, 158-165, 213-218 and vector_nd = 4).
struct LimbExtras {
    const float *jomps;     // [n, 2, H, W] jitter-offset maps at decode resolution, or nullptr
    int vector_nd;          // 2, or 4 for cat_flip_offs offsets ([n, 4L, H, W])
    int use_jitter;         // --use-jitter-offset
    HeadSource scale_lr;    // keypoint-scale maps [.., C, h, w] (fused path; else `scales` at decode resolution)
    HeadSource jitter_lr;   // jitter-offset maps [.., 2, h, w] (fused path; else `jomps`)
};

// What K2 hands to K3 besides the limb table (og_prep.cuh); prep == nullptr: scoring only.
struct PrepOut {
    int32_t *prep;                  // [n, L, K + 1]
    float4 *rec;                    // [n, L, K, 3]
    int32_t *cnt;                   // [n, L]
    float dist_max;
    int use_scale;
    int32_t *clear_word;            // zeroed by the kernel (K3's row allocator), or nullptr
};

// `offs` = materialised full-resolution offsets, or nullptr with `lowres` set.
int launch_limb_score(const float *det_score, const int32_t *det_index, const float *offs,
                      const OffsetSource *lowres, const FlipTablesDev *flips, const float *scales,
                      const LimbExtras *extras, int n, int c, int l, int k, int h, int w,
                      const SkeletonDev &sk, float thre_hmp, float min_len, float resize_factor,
                      float *out_limbs, const PrepOut *prep, cudaStream_t s);

struct ChannelPerm {
    int32_t src[128];
};
// out[n, c] = (a[n, c] + sign * flip_W(b[N + n, perm[c]])) / 2, sign = -1 on even channels if
// negate_even (flip fusion of heat / scale / jitter maps, factory.py:101-113, 141-144)
int launch_flip_average(const float *in2n, float *out, int n, int ch, int h, int w,
                        const ChannelPerm &perm, bool negate_even, cudaStream_t s);
// cat_flip_offs branch (factory.py:115-127): out [n, 4L, h, w] = (x, y, x_flip, y_flip) per limb
int launch_flip_cat_offsets(const float *off2n, float *out, int n, int l, int h, int w,
                            const ChannelPerm &limb_flip, const ChannelPerm &reserved, cudaStream_t s);

bool fused_supported(int n, int c, int scale, int h, int w);
// scratch of the fused K1: floats of the 4 x 4-cell activity map, ints of the block work list
void fused_scratch(int n, int c, int h, int w, int scale, size_t *flag_bytes, size_t *list_ints);
// block_flag: fused_scratch() bytes, ALL ZERO on entry (the kernels leave them zero again);
// block_list: fused_scratch() ints, n_active: one int
// `n` images starting at hmp; the mirrored copy of image i is image n_total + i (flip only)
// `clear_first`: zero the candidate counters / the active-block counter with memsets before the
// kernels (a caller whose select pass runs on ANOTHER stream); otherwise they must be zero on
// entry (launch_select_topk leaves them so).
// Channels-last heat maps: the activity scan transposes them, flip-fused, into `nhwc_heat`
// (dense float32 [n][c][h][w], ignored for planar maps), and the block kernel reads that.
int launch_fused_candidates(const MapView &hmp, const FlipTablesDev &flips, int n, int n_total, int c, int h, int w,
                            int scale, bool cubic, bool flip, float thre, uint32_t *cand_count,
                            uint64_t *cand_keys, uint8_t *block_flag, int32_t *block_list,
                            int32_t *n_active, float *nhwc_heat, int sm_count, bool clear_first,
                            cudaStream_t s, int64_t *launches);

// Network-resolution planes plane_list[0 .. count) (plane = image * C + channel) of `hmp` (either
// layout) as dense float32, averaged with their mirrored partners when `flip` (factory.py:101-106):
// the input of the exact per-plane redo of a fused decode.  `n` = images of the call (the mirrored
// copy of image i is image n + i).
int launch_fuse_planes(const MapView &hmp, const FlipTablesDev &flips, int n, int c, int h, int w, bool flip,
                       const int32_t *plane_list, int count, float *out, cudaStream_t s);

// optional second output of K3: result rows back-projected into the original image frames
struct CocoOut {
    const double *frames;       // [images of the call][4] offset_x, offset_y, scale_x, scale_y; nullptr = off
    float *keypoints;           // [capacity_rows][3 C]  x, y, flag
    double *scores;             // [capacity_rows]
    int32_t *images;            // [capacity_rows] image index within the call
    int image0;                 // index of this launch's first image within the call
};

struct GroupLaunch {
    int n, c, l, k;
    SkeletonDev sk;
    float dist_max;
    int use_scale;
    double person_thre;
    int sort_dim;
    int warp_rows;              // person-table rows of the one-warp-per-image kernel (0 = skip it)
    float *slab;                // the CTA kernel's person tables, one per image
    size_t slab_stride;         // floats between images, multiple of 4
    int32_t *prep;              // group_prep_ints() ints: kept limb rows per (image, limb)
    float4 *rec;                // group_rec_vec4() float4: the kept rows themselves, compacted
    int32_t *cnt;               // [n, L] kept rows per (image, limb)
    int32_t *redo;              // [n] images the warp kernel handed to the CTA kernel
    CocoOut coco;
    int32_t *lazy_flag;         // nullptr: the CTA kernel always follows the warp kernel (early-exit CTAs);
                                // else the warp kernel sets *lazy_flag when an image needs it and the
                                // caller runs launch_group_redo after looking at the flag
};
int read_k3_profile(unsigned long long *out16, bool reset);
size_t group_smem_bytes(const GroupLaunch &g);
size_t group_warp_smem_bytes(const GroupLaunch &g);
size_t group_prep_ints(const GroupLaunch &g);
size_t group_rec_vec4(const GroupLaunch &g);
int prepare_group_kernel(size_t smem_bytes, size_t warp_smem_bytes);
// `prepared`: prep / rec / cnt already hold the rows (K2 wrote them); else the stand-alone
// prepare kernel runs first.  *out_total must be zero on entry.
int launch_group(const GroupLaunch &g, const float *limbs, bool prepared, float *out_poses,
                 int capacity_rows, int32_t *out_offset, int32_t *out_count, int32_t *out_total,
                 cudaStream_t s, int64_t *launches);

// the CTA kernel for the images the warp kernel flagged in g.redo (all images when warp_rows == 0)
int launch_group_redo(const GroupLaunch &g, const float *limbs, float *out_poses, int capacity_rows,
                      int32_t *out_offset, int32_t *out_count, int32_t *out_total, cudaStream_t s,
                      int64_t *launches);

int launch_scored_offset(const float *hmp, const float *off, int n, int c, int l, int h, int w,
                         int ksize, const SkeletonDev &sk, float *out, cudaStream_t s);
int launch_flip_fuse(const float *hmp2n, const float *off2n, const FlipTablesDev &flips,
                     int n, int c, int l, int h, int w, float *out_hmp, float *out_off,
                     cudaStream_t s);
int launch_resize(const float *in, float *out, int planes, int h, int w, int scale, int mode,
                  cudaStream_t s);

}  // namespace og
