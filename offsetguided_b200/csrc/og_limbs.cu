// K2 — limb candidate scoring (reference decoder/collect.py:100-233).
//
// One CTA per (limb type, image).  The K to-joint candidates are staged in shared
// memory; thread k owns from-candidate k: it gathers the guiding offset at its
// peak pixel, adds it to the peak position, scans the K to-candidates for the
// nearest one (first index wins ties, exactly like Tensor.min), and writes the 13
// limb columns.  Everything is float32 with the reference's rounding sequence:
// separate multiply / add where eager torch runs separate kernels, and
// sqrt(fma(dy, dy, dx*dx)) for Tensor.norm over an (x, y) pair (probed against
// ATen's CPU kernel).  ~40 eager launches of the reference collapse into this one.
//
// The nearest to-candidate is found on SQUARED distances (no square root in the K-long
// dependent chain): sqrt is monotonic and correctly rounded, so min(sqrt(d2)) = sqrt(min(d2));
// Tensor.min's first-index rule is then applied to the rounded distances themselves, which
// only the few candidates within 2^-20 of the minimum have to be re-evaluated for.
//
// The same CTA then runs the row-only half of the grouping step for its K rows (og_prep.cuh:
// gate, sort, best row per to-joint id), so K3 starts from compacted kept rows.
#include "og_common.cuh"
#include "og_interp.cuh"
#include "og_prep.cuh"

namespace og {

namespace {

struct ToCand {
    float x, y, score, scale;
    int32_t index;
};

__device__ __forceinline__ float norm2(float dx, float dy) {
    return __fsqrt_rn(__fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
}

// Value at full-resolution pixel (X, Y) of a map that is still at network resolution: x S
// interpolation on the fly (bilinear or bicubic, ATen's taps and accumulation order, og_interp.cuh),
// optionally fused with the flip-test combination of plane `a` (original image) and plane `b`
// (mirrored image, read right-to-left) — bit-identical to gathering from the materialised
// flip_augment + F.interpolate(scale_factor = S) map.  Cell (y, x) of a plane is `pixel_stride`
// elements after cell (y, x - 1): 1 for planar maps, the packed channel count for channels-last.
enum FlipMode { kFlipNone = 0, kFlipAverage = 1, kFlipPartnerOnly = 2 };

template <typename T>
__device__ __forceinline__ float sample_lowres(const T *a, const T *b, int mode, bool negate_b, int h, int w,
                                               size_t pixel_stride, int scale, bool cubic, int X, int Y) {
    auto at = [&](int yy, int xx) {
        if (mode == kFlipNone) return load_cell(a + (size_t)(yy * w + xx) * pixel_stride);
        float m = load_cell(b + (size_t)(yy * w + (w - 1 - xx)) * pixel_stride);
        if (negate_b) m = -m;
        if (mode == kFlipPartnerOnly) return m;
        return __fmul_rn(__fadd_rn(load_cell(a + (size_t)(yy * w + xx) * pixel_stride), m), 0.5f);
    };
    if (scale == 1) return at(Y, X);
    const float inv = 1.0f / (float)scale;
    int ix[4], iy[4];
    float wx[4], wy[4];
    const int taps = axis_taps(X, w, inv, cubic, ix, wx);
    axis_taps(Y, h, inv, cubic, iy, wy);
    if (!cubic) {
        const float r0 = combine2(at(iy[0], ix[0]), at(iy[0], ix[1]), wx[0], wx[1]);
        const float r1 = combine2(at(iy[1], ix[0]), at(iy[1], ix[1]), wx[0], wx[1]);
        return combine2(r0, r1, wy[0], wy[1]);
    }
    float rows[4];
    for (int j = 0; j < taps; ++j)
        rows[j] = combine4(at(iy[j], ix[0]), at(iy[j], ix[1]), at(iy[j], ix[2]), at(iy[j], ix[3]), wx[0], wx[1],
                           wx[2], wx[3]);
    return combine4(rows[0], rows[1], rows[2], rows[3], wy[0], wy[1], wy[2], wy[3]);
}

// Guiding offset (component comp of limb l) at full-resolution pixel (X, Y) from the network-
// resolution offset maps.  comp 0, 1: the flip-test average (factory.py:128-139), or the original
// alone when `cat` (cat_flip_offs, factory.py:115-127); comp 2, 3 (cat only): the mirrored copy's
// vector, x negated; limbs that are their own mirror image keep the original either way.
template <typename T>
__device__ __forceinline__ float sample_offset_t(const OffsetSource &src, const FlipTablesDev &ft, int img, int l,
                                                 int comp, bool cat, int X, int Y) {
    const T *base = static_cast<const T *>(src.maps.ptr);
    const int c2 = comp & 1;
    const T *a = base + (size_t)img * src.maps.image_stride + (size_t)(2 * l + c2) * src.maps.plane_stride;
    const bool mirrored = src.flip && !((ft.reserved >> l) & 1ull);
    const T *b = mirrored ? base + (size_t)(src.n + img) * src.maps.image_stride +
                                (size_t)(2 * (int)ft.limb[l] + c2) * src.maps.plane_stride
                          : nullptr;
    int mode = kFlipNone;
    if (mirrored) mode = cat ? (comp >= 2 ? kFlipPartnerOnly : kFlipNone) : kFlipAverage;
    return sample_lowres(a, b, mode, c2 == 0, src.h, src.w, src.maps.pixel_stride, src.scale, false, X, Y);
}

__device__ __forceinline__ float sample_offset(const OffsetSource &src, const FlipTablesDev &ft, int img, int l,
                                               int comp, bool cat, int X, int Y) {
    if (src.maps.dtype == OG_DTYPE_BF16) return sample_offset_t<__nv_bfloat16>(src, ft, img, l, comp, cat, X, Y);
    if (src.maps.dtype == OG_DTYPE_F16) return sample_offset_t<__half>(src, ft, img, l, comp, cat, X, Y);
    return sample_offset_t<float>(src, ft, img, l, comp, cat, X, Y);
}

// Channel ch of an optional head (keypoint scales: channels = C, mirrored partner ft.kp[ch],
// factory.py:141-144; jitter offsets: channels = 2, partner = the same channel with x negated,
// factory.py:109-113) at full-resolution pixel (X, Y).
__device__ __forceinline__ float sample_head(const HeadSource &hs, const OffsetSource &src, int img, int channels,
                                             int ch, int partner, bool negate_partner, int X, int Y) {
    const size_t hw = (size_t)hs.h * hs.w;
    const float *a = hs.ptr + ((size_t)img * channels + ch) * hw;
    const float *b = src.flip ? hs.ptr + ((size_t)(src.n + img) * channels + partner) * hw : nullptr;
    return sample_lowres(a, b, src.flip ? kFlipAverage : kFlipNone, negate_partner, hs.h, hs.w, (size_t)1, hs.scale,
                         hs.cubic != 0, X, Y);
}

// Tensor.norm over 4 components as ATen's CPU kernel evaluates it (probed) is a plain left-to-right
// sum of squares without fused multiply-add: sq4 below.

// squared distances as Tensor.norm accumulates them before the root
__device__ __forceinline__ float sq2(float dx, float dy) { return __fmaf_rn(dy, dy, __fmul_rn(dx, dx)); }
__device__ __forceinline__ float sq4(float a, float b, float c, float d) {
    float acc = __fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b));
    acc = __fadd_rn(acc, __fmul_rn(c, c));
    return __fadd_rn(acc, __fmul_rn(d, d));
}

template <bool kFour, int KMAX>
__global__ void __launch_bounds__(KMAX)
limb_score_kernel(const float *__restrict__ det_score, const int32_t *__restrict__ det_index,
                  const float *__restrict__ offs, OffsetSource src, FlipTablesDev ft,
                  const float *__restrict__ scales, LimbExtras ex, int C, int L, int K, int H, int W,
                  SkeletonDev sk, float thre_hmp, float min_len, float resize_factor,
                  float *__restrict__ out_limbs, PrepOut po) {
    __shared__ ToCand s_to[KMAX];
    __shared__ PrepShared<KMAX> s_prep;
    const int l = blockIdx.x;
    const int n = blockIdx.y;
    const int jf = sk.from[l], jt = sk.to[l];
    const long long HW = (long long)H * W;
    const int k = threadIdx.x;                     // blockDim.x >= K: one candidate pair per thread
    if (po.clear_word != nullptr && l == 0 && n == 0 && k == 0) *po.clear_word = 0;

    // candidate k of channel j: position, score; sub-threshold candidates (and the
    // empty slots K1 leaves behind, index -1) are moved 100000 px off the image
    // (collect.py:253, integer arithmetic before the float conversion)
    auto candidate = [&](int j, int kk, float &x, float &y, float &s, int32_t &idx) {
        const size_t at = ((size_t)n * C + j) * K + kk;
        s = det_score[at];
        idx = det_index[at];
        int xi = 0, yi = 0;
        if (idx >= 0) {
            yi = idx / W;
            xi = idx - yi * W;
        }
        if (s < thre_hmp) {
            xi -= 100000;
            yi -= 100000;
        }
        x = (float)xi;
        y = (float)yi;
    };

    float row[OG_LIMB_COLS];
#pragma unroll
    for (int i = 0; i < OG_LIMB_COLS; ++i) row[i] = 0.0f;
    float x1 = 0.f, y1 = 0.f, s1 = 0.f;
    int32_t idx1 = -1;
    if (k < K) {
        ToCand t;
        candidate(jt, k, t.x, t.y, t.score, t.index);
        candidate(jf, k, x1, y1, s1, idx1);
        t.scale = 4.0f;                                              // collect.py:120
        if (t.index >= 0) {
            if (scales != nullptr)
                t.scale = __ldg(scales + ((size_t)n * C + jt) * HW + t.index);   // collect.py:114
            else if (ex.scale_lr.ptr != nullptr)
                t.scale = sample_head(ex.scale_lr, src, n, C, jt, ft.kp[jt], false, t.index % W, t.index / W);
        }
        s_to[k] = t;
    }
    // the guiding offset of this thread's from-candidate (global / PCIe gathers: issued before
    // the barrier so that they overlap the staging of the to-candidates)
    float ox = 0.0f, oy = 0.0f, ox2 = 0.0f, oy2 = 0.0f, scale1 = 4.0f;
    if (k < K && idx1 >= 0) {
        if (offs != nullptr) {
            const int nd = kFour ? 4 : 2;
            const float *o = offs + ((size_t)n * nd * L + nd * l) * HW + idx1;   // collect.py:143-147
            ox = __ldg(o);
            oy = __ldg(o + HW);
            if (kFour) {
                ox2 = __ldg(o + 2 * HW);
                oy2 = __ldg(o + 3 * HW);
            }
        } else {
            const int py = idx1 / W, px = idx1 - py * W;
            ox = sample_offset(src, ft, n, l, 0, kFour, px, py);
            oy = sample_offset(src, ft, n, l, 1, kFour, px, py);
            if (kFour) {
                ox2 = sample_offset(src, ft, n, l, 2, true, px, py);
                oy2 = sample_offset(src, ft, n, l, 3, true, px, py);
            }
        }
        if (scales != nullptr)
            scale1 = __ldg(scales + ((size_t)n * C + jf) * HW + idx1);
        else if (ex.scale_lr.ptr != nullptr)
            scale1 = sample_head(ex.scale_lr, src, n, C, jf, ft.kp[jf], false, idx1 % W, idx1 / W);
    }
    __syncthreads();

    if (k < K) {
        float gx = __fadd_rn(x1, __fmul_rn(ox, resize_factor));               // collect.py:152
        float gy = __fadd_rn(y1, __fmul_rn(oy, resize_factor));
        const float gx2 = __fadd_rn(x1, __fmul_rn(ox2, resize_factor));
        const float gy2 = __fadd_rn(y1, __fmul_rn(oy2, resize_factor));
        // jitter-offset component `comp` at decode-resolution pixel (row py, column px)
        const bool have_jitter = ex.jomps != nullptr || ex.jitter_lr.ptr != nullptr;
        auto jitter_at = [&](int comp, int px, int py) {
            if (ex.jomps != nullptr) return __ldg(ex.jomps + ((size_t)n * 2 + comp) * HW + (size_t)py * W + px);
            return sample_head(ex.jitter_lr, src, n, 2, comp, comp, comp == 0, px, py);
        };
        if (have_jitter && ex.use_jitter && !kFour) {
            // jitter refinement of the guided point (collect.py:158-165), including the
            // reference's [x, y]-as-[row, col] indexing; .int() truncates toward zero.
            // (The reference raises IndexError when x >= H; such points are left unrefined.)
            const int xi = (int)gx, yi = (int)gy;
            if (xi >= 0 && xi < W && yi >= 0 && yi < H && xi < H && yi < W) {
                gx = __fadd_rn(gx, jitter_at(0, yi, xi));         // row xi, column yi
                gy = __fadd_rn(gy, jitter_at(1, yi, xi));
            }
        }
        auto sq_to = [&](int m) {
            const float dx = __fsub_rn(gx, s_to[m].x), dy = __fsub_rn(gy, s_to[m].y);
            if (!kFour) return sq2(dx, dy);
            return sq4(dx, dy, __fsub_rn(gx2, s_to[m].x), __fsub_rn(gy2, s_to[m].y));
        };
        // pass 1 (collect.py:171-177): the smallest squared distance; `<` skips a NaN candidate
        // and keeps a NaN first one, like the rounded-distance scan it replaces
        float best2 = sq_to(0);
        for (int m = 1; m < K; ++m) {
            const float d2 = sq_to(m);
            if (d2 < best2) best2 = d2;
        }
        const float best = __fsqrt_rn(best2);
        // pass 2: Tensor.min returns the FIRST index of the smallest ROUNDED distance.  Distinct
        // squared distances within a few ulp can round to the same root, so every candidate
        // within 2^-20 (relative) of the minimum is re-evaluated exactly.
        const float window = __fmul_rn(best2, 1.00000095367431640625f);
        int best_m = 0;
        for (int m = 0; m < K; ++m) {
            const float d2 = sq_to(m);
            if (d2 <= window && __fsqrt_rn(d2) == best) {
                best_m = m;
                break;
            }
        }
        const ToCand t = s_to[best_m];
        const float len = fmaxf(norm2(__fsub_rn(x1, t.x), __fsub_rn(y1, t.y)), min_len);   // :204
        const float score = __fmul_rn(__fmul_rn(s1, t.score), expf(__fdiv_rn(-best, len)));  // :208
        const long long g1 = (long long)idx1 + (long long)jf * HW;             // collect.py:198-199
        const long long g2 = (long long)t.index + (long long)jt * HW;

        float x1o = x1, y1o = y1, x2o = t.x, y2o = t.y;
        if (have_jitter && ex.use_jitter) {        // collect.py:213-218
            if (idx1 >= 0) {
                x1o = __fadd_rn(x1o, jitter_at(0, idx1 % W, idx1 / W));
                y1o = __fadd_rn(y1o, jitter_at(1, idx1 % W, idx1 / W));
            }
            if (t.index >= 0) {
                x2o = __fadd_rn(x2o, jitter_at(0, t.index % W, t.index / W));
                y2o = __fadd_rn(y2o, jitter_at(1, t.index % W, t.index / W));
            }
        }
        row[0] = x1o;                                                   // collect.py:223-233
        row[1] = y1o;
        row[2] = s1;
        row[3] = x2o;
        row[4] = y2o;
        row[5] = t.score;
        row[6] = __ll2float_rn(g1);
        row[7] = __ll2float_rn(g2);
        row[8] = best;
        row[9] = len;
        row[10] = score;
        row[11] = scale1;
        row[12] = t.scale;
        float *o = out_limbs + (((size_t)n * L + l) * K + k) * OG_LIMB_COLS;
#pragma unroll
        for (int i = 0; i < OG_LIMB_COLS; ++i) o[i] = row[i];
    }
    if (po.prep != nullptr) {
        const size_t inst = (size_t)n * L + l;
        prepare_limb_rows(row, k, K, po.dist_max, po.use_scale, s_prep, po.prep + inst * (K + 1),
                          po.rec + inst * K * 3, po.cnt + inst);
    }
}

}  // namespace

int launch_limb_score(const float *det_score, const int32_t *det_index, const float *offs,
                      const OffsetSource *lowres, const FlipTablesDev *flips, const float *scales,
                      const LimbExtras *extras, int n, int c, int l, int k, int h, int w,
                      const SkeletonDev &sk, float thre_hmp, float min_len, float resize_factor,
                      float *out_limbs, const PrepOut *prep, cudaStream_t s) {
    if (n == 0) return OG_OK;
    const int threads = k <= 32 ? 32 : (k <= 64 ? 64 : 128);
    dim3 grid(l, n);
    OffsetSource src = {};
    if (lowres) src = *lowres;
    FlipTablesDev ft = {};
    if (flips) ft = *flips;
    LimbExtras ex = {};
    ex.vector_nd = 2;
    if (extras) ex = *extras;
    PrepOut po = {nullptr, nullptr, nullptr, 0.0f, 0, nullptr};
    if (prep) po = *prep;
#define OG_LAUNCH_K2(FOUR, KMAX)                                                                                  \
    do {                                                                                                          \
        prefer_chain_carveout<limb_score_kernel<FOUR, KMAX>>();                                                   \
        limb_score_kernel<FOUR, KMAX><<<grid, KMAX, 0, s>>>(det_score, det_index, offs, src, ft, scales, ex, c,   \
                                                            l, k, h, w, sk, thre_hmp, min_len, resize_factor,     \
                                                            out_limbs, po);                                       \
    } while (0)
    const bool four = ex.vector_nd == 4;
    if (threads == 32) {
        if (four) OG_LAUNCH_K2(true, 32); else OG_LAUNCH_K2(false, 32);
    } else if (threads == 64) {
        if (four) OG_LAUNCH_K2(true, 64); else OG_LAUNCH_K2(false, 64);
    } else {
        if (four) OG_LAUNCH_K2(true, 128); else OG_LAUNCH_K2(false, 128);
    }
#undef OG_LAUNCH_K2
    OG_CUDA_TRY(cudaGetLastError());
    return OG_OK;
}

}  // namespace og
