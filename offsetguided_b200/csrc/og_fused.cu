// K1f — flip fusion + x S resize + 3x3 NMS + threshold fused into one pass over the
// NETWORK-RESOLUTION heat maps (SURVEY.md 8f-1).
//
// The reference materialises the x4 bicubic map (decoder/factory.py:74-75, 27.9 MB per
// image written, then re-read ~6 times by hmp_NMS / topk).  Here the full-resolution map is
// never written; HBM traffic is C*h*w*4 bytes per image (1.74 MB instead of 55.7 MB).
//
// Threshold first, at network resolution: an interpolated value is bounded by
// (sum |wx|)(sum |wy|) max|taps| <= 1.375^2 max|taps| for the A = -0.75 cubic (1 for bilinear),
// so a region whose taps are all below thre / kBound cannot hold a candidate.  Three kernels:
//
//   amax_scan_kernel    streams the maps once (128-bit loads, 8 rows in flight per thread) — the
//                       only pass that touches all of the input, HBM-bound.  A BLOCK is
//                       (32 / S) x 8 cells = 32 x 8S full-resolution pixels; a cell that can reach
//                       thre (2 % of them) flags the blocks whose cells or tap halo it overlaps;
//   block_list_kernel   compacts the flagged blocks into a work list (and clears the flags);
//   fused_block_kernel  warps stride over the work list, ONE WARP PER BLOCK, one lane per
//                       full-resolution column.  The block's cells (+halo, averaged with the
//                       mirrored copy when flip-testing, prefetched one block ahead into registers)
//                       go to a per-warp shared tile; each lane interpolates its column along x
//                       one tile row at a time into a sliding (TAPS + 1)-row register window and
//                       walks down the 8S rows with one 4-tap (2-tap) combine per pixel in ATen's
//                       accumulation order, so values are bit-identical to the materialised map.
//                       Interpolation weights depend on the phase (pixel mod S) only, so they
//                       live in registers for the lifetime of the warp.  A row in which some lane
//                       reaches thre runs the 3x3 test with lane shuffles; the pixel ring outside
//                       the block is evaluated on demand.  The cell-row loop is deliberately NOT
//                       unrolled: 8S rows of straight-line code (64 KB) thrash the instruction
//                       cache and run 3x slower.
// Skipping is provably lossless (kBound leaves 3 % for rounding); nothing else is skipped.
#include "og_common.cuh"
#include "og_interp.cuh"

#include <algorithm>

namespace og {

namespace {

#ifndef OG_K1F_MIN_CTAS
#define OG_K1F_MIN_CTAS 4
#endif
constexpr int kFusedThreads = 256;
constexpr int kScanThreads = 256;
constexpr int kBlockCellsH = 8;       // cell rows of a block
constexpr int kSub = 4;               // cells per scan thread along x (one vector load); 2 x kSub rows
constexpr unsigned kFull = 0xffffffffu;

__device__ __forceinline__ float4 ldg_stream4(const float *p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}

// four consecutive cells with one streaming load (16 / 8 bytes)
__device__ __forceinline__ float4 load_cells4(const float *p) { return ldg_stream4(p); }
__device__ __forceinline__ float4 load_cells4(const __nv_bfloat16 *p) {
    unsigned lo, hi;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "l"(p));
    return make_float4(__uint_as_float(lo << 16), __uint_as_float(lo & 0xffff0000u),
                       __uint_as_float(hi << 16), __uint_as_float(hi & 0xffff0000u));
}

__device__ __forceinline__ float4 load_cells4(const __half *p) {
    unsigned lo, hi;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "l"(p));
    const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&lo));
    const float2 b = __half22float2(*reinterpret_cast<const __half2 *>(&hi));
    return make_float4(a.x, a.y, b.x, b.y);
}

// |v| >= 0: the IEEE bit pattern orders like the value, and NaN sorts above everything,
// which keeps such regions active
__device__ __forceinline__ unsigned abs_bits(float v) { return __float_as_uint(fabsf(v)); }

// ---- pass A: activity flags ----------------------------------------------------
// one thread per (plane, 8-row band, 4-cell column group); 32-bit index arithmetic (the host splits
// calls of more than 2^31 threads into several launches over `plane0`)
template <typename T, bool kFlip, bool kVec>
__global__ void __launch_bounds__(kScanThreads)
amax_scan_kernel(const T *__restrict__ hmp, size_t img_stride, const FlipTablesDev ft,
                 int N, int C, int h, int w, int bw_shift, int halo, float limit,
                 uint8_t *__restrict__ block_flag, int plane0, int planes, int per_plane) {
    const unsigned idx = blockIdx.x * (unsigned)kScanThreads + threadIdx.x;
    const unsigned pl = idx / (unsigned)per_plane;
    if (pl >= (unsigned)planes) return;
    const int local = (int)(idx - pl * (unsigned)per_plane);
    const int sxs = (w + kSub - 1) / kSub;
    const int band = local / sxs, sx = local - band * sxs;
    const int y0 = band * 2 * kSub, x0 = sx * kSub;
    const int block_w = 1 << bw_shift;
    const int bxs = (w + block_w - 1) >> bw_shift, bys = (h + kBlockCellsH - 1) / kBlockCellsH;
    {
        const int plane = plane0 + (int)pl;
        const int n = plane / C, c = plane - n * C;
        const T *a = hmp + (size_t)n * img_stride + (size_t)c * h * w;
        const T *b = nullptr;
        if (kFlip) b = hmp + (size_t)(N + n) * img_stride + (size_t)ft.kp[c] * h * w;
        uint8_t *flags = block_flag + (size_t)plane * bys * bxs;
        // Cells [xa, xb] of row y can reach the threshold (rare): flag every work block whose cells
        // or tap halo they overlap.  Plain byte stores of the same value from many threads are benign.
        auto flag_blocks = [&](int xa, int xb, int y) {
            const int bx_lo = max(xa - halo, 0) >> bw_shift, bx_hi = min((xb + halo) >> bw_shift, bxs - 1);
            const int by_lo = max(y - halo, 0) / kBlockCellsH, by_hi = min((y + halo) / kBlockCellsH, bys - 1);
            for (int by = by_lo; by <= by_hi; ++by)
                for (int bx = bx_lo; bx <= bx_hi; ++bx) flags[by * bxs + bx] = 1;
        };
        if (kVec) {
            // two batches of kSub rows: 4 (8 with the mirrored copy) independent 128-bit loads in
            // flight per thread keep the register count low enough for full occupancy
#pragma unroll 1
            for (int r0 = 0; r0 < 2 * kSub; r0 += kSub) {
                float4 va[kSub], vb[kSub];
#pragma unroll
                for (int r = 0; r < kSub; ++r) {
                    const int y = min(y0 + r0 + r, h - 1);     // rows below the image repeat the last one
                    va[r] = load_cells4(a + (size_t)y * w + x0);
                    if (kFlip) vb[r] = load_cells4(b + (size_t)y * w + (w - kSub - x0));
                }
                auto fused_row = [&](int r) {
                    float4 f = va[r];
                    if (kFlip) {             // (orig + flip_W(flipped)[kp_flip]) / 2, factory.py:101-106
                        f.x = __fmul_rn(__fadd_rn(f.x, vb[r].w), 0.5f);
                        f.y = __fmul_rn(__fadd_rn(f.y, vb[r].z), 0.5f);
                        f.z = __fmul_rn(__fadd_rn(f.z, vb[r].y), 0.5f);
                        f.w = __fmul_rn(__fadd_rn(f.w, vb[r].x), 0.5f);
                    }
                    return f;
                };
                // the streaming test: one bit per row, no branch; the rows that pass (2 % of the
                // cells) are looked at again in ONE divergent region per batch
                unsigned hot = 0u;
#pragma unroll
                for (int r = 0; r < kSub; ++r) {
                    const float4 f = fused_row(r);
                    const unsigned q = max(max(abs_bits(f.x), abs_bits(f.y)), max(abs_bits(f.z), abs_bits(f.w)));
                    if (!(__uint_as_float(q) < limit) && y0 + r0 + r < h) hot |= 1u << r;   // NaN is not below: stays active
                }
                if (hot != 0u) {
#pragma unroll
                    for (int r = 0; r < kSub; ++r) {
                        if (!((hot >> r) & 1u)) continue;
                        const float4 f = fused_row(r);
                        const bool c0 = !(fabsf(f.x) < limit), c1 = !(fabsf(f.y) < limit), c2 = !(fabsf(f.z) < limit),
                                   c3 = !(fabsf(f.w) < limit);
                        const int first = c0 ? 0 : (c1 ? 1 : (c2 ? 2 : 3));
                        const int last = c3 ? 3 : (c2 ? 2 : (c1 ? 1 : 0));
                        flag_blocks(x0 + first, x0 + last, y0 + r0 + r);
                    }
                }
            }
        } else {
            for (int r = 0; r < 2 * kSub; ++r) {
                const int y = y0 + r;
                if (y >= h) break;
                for (int j = 0; j < kSub; ++j) {
                    const int x = x0 + j;
                    if (x >= w) break;
                    float v = load_cell(a + (size_t)y * w + x);
                    if (kFlip) v = __fmul_rn(__fadd_rn(v, load_cell(b + (size_t)y * w + (w - 1 - x))), 0.5f);
                    if (!(fabsf(v) < limit)) flag_blocks(x, x, y);
                }
            }
        }
    }
}

// ---- pass A for channels-last maps: transposing activity scan ------------------------
// Cell (y, x) of channel c is at (y * w + x) * P + c (P >= C: the channel count of the packed
// tensor), so a plane's cells are P elements apart and a block kernel gathering them would touch
// a 32-byte sector per cell.  This pass is the only one over the channels-last heat channels: it
// reads each pixel's C channels (with flip-test also the mirrored image's pixel w - 1 - x, channel
// kp[c]), writes the fused values as dense float32 planes `out` [n][C][h][w] for the block kernel,
// and flags exactly the blocks amax_scan_kernel would flag on those planes.
// One CTA per (image, 8-row band, 32-pixel column group).  A row's 32 x C values are loaded with
// consecutive threads on consecutive channels of consecutive pixels (coalesced along the pixel run),
// staged in shared memory, and written as 32-cell runs of each plane.
constexpr int kNhwcPixels = 32;
constexpr int kNhwcThreads = 256;

template <typename T, bool kFlip>
__global__ void __launch_bounds__(kNhwcThreads)
amax_scan_nhwc_kernel(const T *__restrict__ hmp, size_t img_stride, size_t pix_stride, const FlipTablesDev ft,
                      int N, int C, int h, int w, int bw_shift, int halo, float limit,
                      uint8_t *__restrict__ block_flag, float *__restrict__ out) {
    __shared__ float s_row[OG_MAX_KEYPOINTS][kNhwcPixels + 1];
    const int gxs = (w + kNhwcPixels - 1) / kNhwcPixels, bands = (h + kBlockCellsH - 1) / kBlockCellsH;
    const unsigned cta = blockIdx.x;
    const int gx = (int)(cta % (unsigned)gxs);
    const int band = (int)((cta / (unsigned)gxs) % (unsigned)bands);
    const int n = (int)(cta / ((unsigned)gxs * (unsigned)bands));
    const int x0 = gx * kNhwcPixels, y0 = band * kBlockCellsH;
    const int px_n = min(kNhwcPixels, w - x0), y_end = min(y0 + kBlockCellsH, h);
    const int block_w = 1 << bw_shift;
    const int bxs = (w + block_w - 1) >> bw_shift, bys = (h + kBlockCellsH - 1) / kBlockCellsH;
    const size_t hw = (size_t)h * w;
    const T *a = hmp + (size_t)n * img_stride;
    const T *b = kFlip ? hmp + (size_t)(N + n) * img_stride : nullptr;
    const int cells = px_n * C;
    for (int y = y0; y < y_end; ++y) {
        for (int i = threadIdx.x; i < cells; i += kNhwcThreads) {
            const int px = i / C, c = i - px * C;
            const int x = x0 + px;
            float v = load_cell(a + ((size_t)y * w + x) * pix_stride + c);
            if (kFlip)                       // (orig + flip_W(flipped)[kp_flip]) / 2, factory.py:101-106
                v = __fmul_rn(__fadd_rn(v, load_cell(b + ((size_t)y * w + (w - 1 - x)) * pix_stride + ft.kp[c])), 0.5f);
            s_row[c][px] = v;
        }
        __syncthreads();
        for (int j = threadIdx.x; j < C * kNhwcPixels; j += kNhwcThreads) {
            const int c = j / kNhwcPixels, px = j - c * kNhwcPixels;
            if (px >= px_n) continue;
            const int x = x0 + px;
            const float v = s_row[c][px];
            const int plane = n * C + c;
            out[(size_t)plane * hw + (size_t)y * w + x] = v;
            if (!(fabsf(v) < limit)) {       // NaN is not below: stays active
                uint8_t *flags = block_flag + (size_t)plane * bys * bxs;
                const int bx_lo = max(x - halo, 0) >> bw_shift, bx_hi = min((x + halo) >> bw_shift, bxs - 1);
                const int by_lo = max(y - halo, 0) / kBlockCellsH, by_hi = min((y + halo) / kBlockCellsH, bys - 1);
                for (int by = by_lo; by <= by_hi; ++by)
                    for (int bx = bx_lo; bx <= bx_hi; ++bx) flags[by * bxs + bx] = 1;
            }
        }
        __syncthreads();
    }
}

// ---- pass B: work list -----------------------------------------------------------
// Compacts the flagged blocks and clears the flags for the next call.
// entry = {plane (image * C + channel), image, block row << 16 | block column,
//          channel | channel of the mirrored map << 16}
__global__ void __launch_bounds__(256)
block_list_kernel(uint8_t *__restrict__ block_flag, const FlipTablesDev ft, int C,
                  int flip, int bxs, int bys, long long total, int4 *__restrict__ block_list,
                  int32_t *__restrict__ n_active) {
    __shared__ int s_warp[8];
    __shared__ int s_base;
    const long long g = (long long)blockIdx.x * 256 + threadIdx.x;
    bool active = false;
    if (g < total) {
        active = block_flag[g] != 0;
        if (active) block_flag[g] = 0;
    }
    // one global atomic per CTA
    const unsigned ballot = __ballot_sync(kFull, active);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) s_warp[warp] = __popc(ballot);
    __syncthreads();
    if (threadIdx.x == 0) {
        int sum = 0;
        for (int i = 0; i < 8; ++i) {
            const int cnt = s_warp[i];
            s_warp[i] = sum;
            sum += cnt;
        }
        s_base = sum ? atomicAdd(n_active, sum) : 0;
    }
    __syncthreads();
    if (active) {
        const int bx = (int)(g % bxs);
        const int by = (int)((g / bxs) % bys);
        const int plane = (int)(g / ((long long)bxs * bys));
        const int n = plane / C, c = plane - n * C;
        const int cb = flip ? (int)ft.kp[c] : c;
        block_list[s_base + s_warp[warp] + __popc(ballot & ((1u << lane) - 1u))] =
            make_int4(plane, n, (by << 16) | bx, c | (cb << 16));
    }
}

// ---- pass C: interpolation + NMS over the active blocks -------------------------------
// value of one full-resolution pixel from the warp's cell tile, generic taps (ring pixels only)
template <int S, bool kCubic, int LW, int HALO>
__device__ __noinline__ float tile_value(const float *lo, int cx0, int cy0, int X, int Y) {
    constexpr int TAPS = kCubic ? 4 : 2;
    const float inv = 1.0f / (float)S;
    float wxs[4], wys[4];
    const int fx = axis_first_tap(X, inv, kCubic, wxs) - (cx0 - HALO);
    const int fy = axis_first_tap(Y, inv, kCubic, wys) - (cy0 - HALO);
    float rows[TAPS];
#pragma unroll
    for (int t = 0; t < TAPS; ++t) {
        const float *row = lo + (fy + t) * LW + fx;
        rows[t] = kCubic ? combine4(row[0], row[1], row[2], row[3], wxs[0], wxs[1], wxs[2], wxs[3])
                         : combine2(row[0], row[1], wxs[0], wxs[1]);
    }
    return kCubic ? combine4(rows[0], rows[1], rows[TAPS - 2], rows[TAPS - 1], wys[0], wys[1], wys[2], wys[3])
                  : combine2(rows[0], rows[1], wys[0], wys[1]);
}

template <typename T, int S, bool kCubic, bool kFlip>
__global__ void __launch_bounds__(kFusedThreads, S <= 4 ? OG_K1F_MIN_CTAS : 3)
fused_block_kernel(const T *__restrict__ hmp, size_t img_stride, int N, int h, int w, float thre,
                   const int4 *__restrict__ block_list,
                   const int32_t *__restrict__ n_active_ptr, uint32_t *__restrict__ cand_count,
                   uint64_t *__restrict__ cand_keys) {
    constexpr int HALO = kCubic ? 2 : 1;
    constexpr int TAPS = kCubic ? 4 : 2;
    constexpr int BW = 32 / S, BH = kBlockCellsH;
    constexpr int LW = BW + 2 * HALO, LH = BH + 2 * HALO;
    constexpr int NL = (LW * LH + 31) / 32;
    constexpr int kWarps = kFusedThreads / 32;
    __shared__ float s_lo[kWarps][LH * LW];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float *lo = s_lo[warp];
    const int W = w * S, H = h * S;
    const int n_active = *n_active_ptr;
    const int stride = gridDim.x * kWarps;
    const float inv = 1.0f / (float)S;

    // Interpolation weights depend on the phase (pixel mod S) only: src = (dst + 0.5) / S - 0.5
    // is exact in float for a power-of-two S.  The one exception is bilinear's clamp of src at 0
    // (pixels < S / 2 from the top / left image border), handled where the taps are combined.
    float wx[4];
    axis_first_tap(lane + 2 * 32, inv, kCubic, wx);
    const int xb_phase = lane / S + ((lane % S) >= S / 2 ? 1 : 0);     // first tap, tile-relative
    float wy[S][TAPS];
#pragma unroll
    for (int p = 0; p < S; ++p) {
        float t4[4];
        axis_first_tap(p + 8 * S, inv, kCubic, t4);
#pragma unroll
        for (int t = 0; t < TAPS; ++t) wy[p][t] = t4[t];
    }

    // cells of a block (+halo), border cells replicated (= ATen's tap clamping), fused with
    // the mirrored copy: (orig + flip_W(flipped)[kp_flip]) / 2   (factory.py:101-106)
    const size_t hw = (size_t)h * w;
    auto load_block = [&](const int4 e, float (&vals)[NL]) {
        const int base_x = (e.z & 0xffff) * BW - HALO, base_y = (e.z >> 16) * BH - HALO;
        const T *a = hmp + (size_t)e.y * img_stride + (size_t)(e.w & 0xffff) * hw;
        const T *b = hmp + (size_t)(N + e.y) * img_stride + (size_t)(e.w >> 16) * hw;
        const bool interior = base_x >= 0 && base_y >= 0 && base_x + LW <= w && base_y + LH <= h;
        if (interior) {                     // warp-uniform: no clamping; 32-bit indices off two bases
            const int ao = base_y * w + base_x;
            const int bo = base_y * w + (w - 1 - base_x);
#pragma unroll
            for (int u = 0; u < NL; ++u) {
                const int i = lane + 32 * u;
                float v = 0.0f;
                if (i < LH * LW) {
                    const int ly = i / LW, lx = i - ly * LW;
                    const int row = ly * w;
                    v = load_cell(a + (ao + row + lx));
                    if (kFlip) v = __fmul_rn(__fadd_rn(v, load_cell(b + (bo + row - lx))), 0.5f);
                }
                vals[u] = v;
            }
        } else {
#pragma unroll
            for (int u = 0; u < NL; ++u) {
                const int i = lane + 32 * u;
                float v = 0.0f;
                if (i < LH * LW) {
                    const int ly = i / LW, lx = i - ly * LW;
                    const int gy = min(max(base_y + ly, 0), h - 1);
                    const int gx = min(max(base_x + lx, 0), w - 1);
                    v = load_cell(a + (gy * w + gx));
                    if (kFlip) v = __fmul_rn(__fadd_rn(v, load_cell(b + (gy * w + (w - 1 - gx)))), 0.5f);
                }
                vals[u] = v;
            }
        }
    };

    float vals[NL];
    int item = blockIdx.x * kWarps + warp;
    int4 blk = make_int4(0, 0, 0, 0), blk_next = blk;
    if (item < n_active) {
        blk = block_list[item];
        load_block(blk, vals);
    }
    for (; item < n_active; item += stride, blk = blk_next) {
        const int plane = blk.x;
        const int cx0 = (blk.z & 0xffff) * BW, cy0 = (blk.z >> 16) * BH;
        const int X0 = cx0 * S, Y0 = cy0 * S;
        const int X = X0 + lane;

        __syncwarp();                       // the previous block's reads of the tile are done
#pragma unroll
        for (int u = 0; u < NL; ++u) {
            const int i = lane + 32 * u;
            if (i < LH * LW) lo[i] = vals[u];
        }
        if (item + stride < n_active) {     // prefetch the next block of this warp into registers
            blk_next = block_list[item + stride];
            load_block(blk_next, vals);
        }
        __syncwarp();

        // This lane's column: tile rows are interpolated along x one at a time (xrow) into a
        // sliding window win[k] = row q + k of the column, k = 0 .. TAPS; the S pixels of cell row q
        // combine win[0 .. TAPS-1] (phase < S / 2) or win[1 .. TAPS] along y.
        const bool clamp_l = !kCubic && X < S / 2;
        const int xb = clamp_l ? 1 : xb_phase;
        const float wx0 = clamp_l ? 1.0f : wx[0], wx1 = clamp_l ? 0.0f : wx[1];
        const bool inside = X < W;             // outside the image: zero padding of the NMS window
        auto xrow = [&](int ly) {
            const float *row = lo + ly * LW + xb;
            const float v = kCubic ? combine4(row[0], row[1], row[2], row[3], wx0, wx1, wx[2], wx[3])
                                   : combine2(row[0], row[1], wx0, wx1);
            return inside ? v : 0.0f;
        };
        float win[TAPS + 1];
        win[0] = 0.0f;
#pragma unroll
        for (int k = 1; k <= TAPS; ++k) win[k] = xrow(k - 1);
        auto ycombine = [&](int first, int p) {        // taps win[first ..], weights of phase p
            return kCubic ? combine4(win[first], win[first + 1], win[first + TAPS - 2], win[first + TAPS - 1],
                                     wy[p][0], wy[p][1], wy[p][TAPS - 2], wy[p][TAPS - 1])
                          : combine2(win[first], win[first + 1], wy[p][0], wy[p][1]);
        };
        const bool clamp_t = !kCubic && Y0 == 0;

        // v[0] = pixel row above cell row q, v[1 .. S] = its S rows, v[S + 1] = the row below
        float v[S + 2];
        v[S] = 0.0f;
        if (Y0 > 0) v[S] = ycombine(1, S - 1);        // last pixel row of the cell row above the block
        v[S + 1] = 0.0f;
        const int valid_q = min(h - cy0, BH + 1);     // cell rows of the image below the block's top
#pragma unroll 1
        for (int q = 0; q < BH && q < valid_q; ++q) {
#pragma unroll
            for (int k = 0; k < TAPS; ++k) win[k] = win[k + 1];
            win[TAPS] = xrow(q + TAPS);
            const bool top = clamp_t && q == 0;    // bilinear rows above src = 0: value = first cell row
            v[0] = v[S];
            v[1] = q == 0 ? (top ? combine2(win[1], win[2], 1.0f, 0.0f) : ycombine(0, 0)) : v[S + 1];
#pragma unroll
            for (int p = 1; p < S; ++p) {
                v[p + 1] = ycombine(p >= S / 2 ? 1 : 0, p);
                if (top && p < S / 2) v[p + 1] = combine2(win[1], win[2], 1.0f, 0.0f);
            }
            // first pixel row of the next cell row; zero padding below the image
            v[S + 1] = q + 1 < valid_q ? ycombine(1, 0) : 0.0f;
            // Threshold and the two vertical neighbours first (this lane's own registers): only a
            // row that holds a vertical maximum above thre — about one row per blob and column —
            // pays for the shuffles, and a cell row without any costs one vote.  fmaxf drops a NaN
            // neighbour like !(neighbour > v) does; thre > 0, so zero padding never passes.
            unsigned mask = 0u;
#pragma unroll
            for (int p = 0; p < S; ++p)
                if (v[p + 1] >= fmaxf(thre, fmaxf(v[p], v[p + 2]))) mask |= 1u << p;
            if (!__any_sync(kFull, mask != 0u)) continue;
#pragma unroll
            for (int p = 0; p < S; ++p) {
                const bool pass = (mask >> p) & 1u;
                if (!__any_sync(kFull, pass)) continue;
                const float vp = v[p], vc = v[p + 1], vn = v[p + 2];
                const float lp = __shfl_up_sync(kFull, vp, 1), lc = __shfl_up_sync(kFull, vc, 1),
                            ln = __shfl_up_sync(kFull, vn, 1);
                const float rp = __shfl_down_sync(kFull, vp, 1), rc = __shfl_down_sync(kFull, vc, 1),
                            rn = __shfl_down_sync(kFull, vn, 1);
                if (pass) {
                    const int Y = Y0 + q * S + p;
                    bool peak = true;
                    if (lane > 0) peak = peak && !(lp > vc) && !(lc > vc) && !(ln > vc);
                    if (lane < 31) peak = peak && !(rp > vc) && !(rc > vc) && !(rn > vc);
                    // ring columns outside the block: evaluated only for a pixel that survived
                    // everything else
                    if (peak && ((lane == 0 && X0 > 0) || (lane == 31 && X + 1 < W))) {
                        const int Xn = lane == 0 ? X - 1 : X + 1;
                        for (int dy = -1; dy <= 1 && peak; ++dy) {
                            if (Y + dy < 0 || Y + dy >= H) continue;
                            peak = !(tile_value<S, kCubic, LW, HALO>(lo, cx0, cy0, Xn, Y + dy) > vc);
                        }
                    }
                    if (peak) {
                        const uint32_t pos = atomicAdd(&cand_count[plane], 1u);
                        if (pos < (uint32_t)kCandCap)
                            cand_keys[(size_t)plane * kCandCap + pos] =
                                make_key(vc + 0.0f, (uint32_t)(Y * W + X));
                    }
                }
            }
        }
    }
}

// resident CTAs per SM of one instantiation (queried once: the answer is a property of the kernel)
template <typename Kernel>
int resident_per_sm(Kernel kernel) {
    int per_sm = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kFusedThreads, 0) != cudaSuccess ||
        per_sm < 1)
        per_sm = 1;
    return per_sm;
}

// CTA waves of the block kernel's grid (2 and 1 measured no faster: profiles/r2_dropped_experiments.txt)
constexpr int kCtaWaves = 4;

template <typename T, int S, bool kCubic, bool kFlip>
int launch_blocks_t(const T *hmp, size_t img_stride, int n_total, int h, int w, float thre,
                    const int4 *block_list, const int32_t *n_active, uint32_t *cand_count,
                    uint64_t *cand_keys, int sm_count, size_t blocks, cudaStream_t s) {
    auto kernel = fused_block_kernel<T, S, kCubic, kFlip>;
    // Warps stride over the work list.  kCtaWaves x the resident CTA count: the per-warp setup
    // (weights) is still amortised over several blocks, but CTAs retire during the kernel, so the
    // high-priority K3 CTAs of the previous call find room instead of waiting for a fully
    // persistent grid to drain.
    static const int per_sm = resident_per_sm(kernel);
    const int grid = (int)std::min<size_t>((blocks + kFusedThreads / 32 - 1) / (kFusedThreads / 32),
                                           (size_t)sm_count * per_sm * kCtaWaves);
    prefer_chain_carveout<fused_block_kernel<T, S, kCubic, kFlip>>();
    kernel<<<grid, kFusedThreads, 0, s>>>(hmp, img_stride, n_total, h, w, thre, block_list, n_active,
                                          cand_count, cand_keys);
    OG_CUDA_TRY(cudaGetLastError());
    return OG_OK;
}

template <typename T, int S>
int launch_blocks_s(const T *hmp, size_t img_stride, int n_total, int h, int w, bool cubic, bool flip,
                    float thre, const int4 *block_list, const int32_t *n_active, uint32_t *cand_count,
                    uint64_t *cand_keys, int sm_count, size_t blocks, cudaStream_t s) {
    if (cubic)
        return flip ? launch_blocks_t<T, S, true, true>(hmp, img_stride, n_total, h, w, thre, block_list, n_active, cand_count, cand_keys, sm_count, blocks, s)
                    : launch_blocks_t<T, S, true, false>(hmp, img_stride, n_total, h, w, thre, block_list, n_active, cand_count, cand_keys, sm_count, blocks, s);
    return flip ? launch_blocks_t<T, S, false, true>(hmp, img_stride, n_total, h, w, thre, block_list, n_active, cand_count, cand_keys, sm_count, blocks, s)
                : launch_blocks_t<T, S, false, false>(hmp, img_stride, n_total, h, w, thre, block_list, n_active, cand_count, cand_keys, sm_count, blocks, s);
}

inline size_t block_count(int n, int c, int h, int w, int scale) {
    const int bw = 32 / scale;
    return (size_t)n * c * ((w + bw - 1) / bw) * ((h + kBlockCellsH - 1) / kBlockCellsH);
}

}  // namespace

bool fused_supported(int n, int c, int scale, int h, int w) {
    if (!(scale == 2 || scale == 4 || scale == 8)) return false;
    return block_count(n, c, h, w, scale) < 0x1fffffffULL && h < 65536 * kBlockCellsH && w < 65536 &&
           (unsigned long long)h * scale * w * scale < 0xffffffffULL;
}

void fused_scratch(int n, int c, int h, int w, int scale, size_t *flag_bytes, size_t *list_ints) {
    *flag_bytes = block_count(n, c, h, w, scale);               // one byte per work block
    *list_ints = 4 * block_count(n, c, h, w, scale);          // int4 entries
}

namespace {
// the activity scan's parameters: log2 of the block width in cells, the tap halo and the cell limit
inline int scan_bw_shift(int scale) { return scale == 2 ? 4 : (scale == 4 ? 3 : 2); }
inline int scan_halo(bool cubic) { return cubic ? 2 : 1; }
inline float scan_limit(float thre, bool cubic) { return thre / (cubic ? 1.95f : 1.001f); }

template <typename T>
int launch_scan_nhwc_t(const T *hmp, size_t img_stride, size_t pix_stride, const FlipTablesDev &kp_flip_dev, int n,
                       int n_total, int c, int h, int w, int scale, bool cubic, bool flip, float thre,
                       uint8_t *block_flag, float *out, cudaStream_t s) {
    const long long ctas = (long long)n * ((w + kNhwcPixels - 1) / kNhwcPixels) *
                           ((h + kBlockCellsH - 1) / kBlockCellsH);
    if (ctas > 0x7fffffffLL) {
        set_error("fused K1: %lld scan CTAs of channels-last maps exceed one launch", ctas);
        return OG_ERR_UNSUPPORTED;
    }
#define OG_SCAN_NHWC(FLIP)                                                                                      \
    (prefer_chain_carveout<amax_scan_nhwc_kernel<T, FLIP>>(),                                                    \
     amax_scan_nhwc_kernel<T, FLIP><<<(unsigned)ctas, kNhwcThreads, 0, s>>>(                                     \
         hmp, img_stride, pix_stride, kp_flip_dev, n_total, c, h, w, scan_bw_shift(scale), scan_halo(cubic),     \
         scan_limit(thre, cubic), block_flag, out))
    if (flip) OG_SCAN_NHWC(true); else OG_SCAN_NHWC(false);
#undef OG_SCAN_NHWC
    OG_CUDA_TRY(cudaGetLastError());
    return OG_OK;
}

// `scan`: run the activity scan over `hmp`; false when the transposing scan already flagged the
// blocks and wrote `hmp` (its dense float32 output)
template <typename T>
int launch_fused_t(const T *hmp, size_t img_stride, const FlipTablesDev &kp_flip_dev, int n, int n_total,
                   int c, int h, int w, int scale, bool cubic, bool flip, float thre,
                   uint32_t *cand_count, uint64_t *cand_keys, uint8_t *block_flag, int32_t *block_list,
                   int32_t *n_active, int sm_count, bool clear_first, bool scan, cudaStream_t s,
                   int64_t *launches) {
    if (clear_first) {
        OG_CUDA_TRY(cudaMemsetAsync(cand_count, 0, sizeof(uint32_t) * (size_t)n * c, s));
        OG_CUDA_TRY(cudaMemsetAsync(n_active, 0, sizeof(int32_t), s));
    }

    const int sxs = (w + kSub - 1) / kSub, bands = (h + 2 * kSub - 1) / (2 * kSub);
    const int per_plane = bands * sxs, planes = scan ? n * c : 0;
    const int planes_per_launch = std::max(1, (int)std::min<long long>(n * c, 0x7fffffffLL / per_plane - 1));
    const int block_w = 32 / scale, halo = scan_halo(cubic);
    const int bw_shift = scan_bw_shift(scale);
    const float limit = scan_limit(thre, cubic);
    // vector loads need whole 4-cell groups and rows aligned to the 4-cell load size (also the
    // rows of the mirrored read and of every image)
    const size_t vec_bytes = 4 * sizeof(T);
    const bool vec = (w % kSub) == 0 && (reinterpret_cast<uintptr_t>(hmp) % vec_bytes) == 0 &&
                     (img_stride * sizeof(T)) % vec_bytes == 0;
#define OG_SCAN(FLIP, VEC)                                                                                     \
    (prefer_chain_carveout<amax_scan_kernel<T, FLIP, VEC>>(),                                                  \
     amax_scan_kernel<T, FLIP, VEC><<<scan_grid, kScanThreads, 0, s>>>(hmp, img_stride, kp_flip_dev, n_total, c, h, \
                                                                      w, bw_shift, halo, limit, block_flag, p0, pn, \
                                                                      per_plane))
    for (int p0 = 0; p0 < planes; p0 += planes_per_launch) {
        const int pn = std::min(planes_per_launch, planes - p0);
        const unsigned scan_grid = (unsigned)(((long long)pn * per_plane + kScanThreads - 1) / kScanThreads);
        if (flip) {
            if (vec) OG_SCAN(true, true); else OG_SCAN(true, false);
        } else {
            if (vec) OG_SCAN(false, true); else OG_SCAN(false, false);
        }
    }
#undef OG_SCAN
    OG_CUDA_TRY(cudaGetLastError());

    const size_t blocks = block_count(n, c, h, w, scale);
    int4 *list4 = reinterpret_cast<int4 *>(block_list);
    prefer_chain_carveout<block_list_kernel>();
    block_list_kernel<<<(unsigned)((blocks + 255) / 256), 256, 0, s>>>(
        block_flag, kp_flip_dev, c, flip ? 1 : 0, (w + block_w - 1) / block_w,
        (h + kBlockCellsH - 1) / kBlockCellsH, (long long)blocks, list4, n_active);
    OG_CUDA_TRY(cudaGetLastError());

    int st;
    switch (scale) {
        case 2: st = launch_blocks_s<T, 2>(hmp, img_stride, n_total, h, w, cubic, flip, thre, list4, n_active, cand_count, cand_keys, sm_count, blocks, s); break;
        case 4: st = launch_blocks_s<T, 4>(hmp, img_stride, n_total, h, w, cubic, flip, thre, list4, n_active, cand_count, cand_keys, sm_count, blocks, s); break;
        default: st = launch_blocks_s<T, 8>(hmp, img_stride, n_total, h, w, cubic, flip, thre, list4, n_active, cand_count, cand_keys, sm_count, blocks, s); break;
    }
    if (st == OG_OK && launches) *launches += 3;
    return st;
}
}  // namespace

int launch_fused_candidates(const MapView &hmp, const FlipTablesDev &kp_flip_dev, int n, int n_total, int c,
                            int h, int w, int scale, bool cubic, bool flip, float thre,
                            uint32_t *cand_count, uint64_t *cand_keys, uint8_t *block_flag,
                            int32_t *block_list, int32_t *n_active, float *nhwc_heat, int sm_count,
                            bool clear_first, cudaStream_t s, int64_t *launches) {
    if (n == 0) return OG_OK;
    if (!fused_supported(n, c, scale, h, w)) {
        set_error("fused K1: scale %d / %d x %d maps are outside the supported range", scale, h, w);
        return OG_ERR_UNSUPPORTED;
    }
    if (hmp.is_channels_last()) {
        // the transposing scan replaces the planar one; the block kernel then runs on its dense
        // float32, already flip-fused output (no mirrored image left to read)
        if (clear_first) {          // before the scan: the counters of an earlier range may still be read
            OG_CUDA_TRY(cudaMemsetAsync(cand_count, 0, sizeof(uint32_t) * (size_t)n * c, s));
            OG_CUDA_TRY(cudaMemsetAsync(n_active, 0, sizeof(int32_t), s));
        }
        int st;
        if (hmp.dtype == OG_DTYPE_BF16)
            st = launch_scan_nhwc_t(static_cast<const __nv_bfloat16 *>(hmp.ptr), hmp.image_stride, hmp.pixel_stride,
                                    kp_flip_dev, n, n_total, c, h, w, scale, cubic, flip, thre, block_flag, nhwc_heat, s);
        else if (hmp.dtype == OG_DTYPE_F16)
            st = launch_scan_nhwc_t(static_cast<const __half *>(hmp.ptr), hmp.image_stride, hmp.pixel_stride,
                                    kp_flip_dev, n, n_total, c, h, w, scale, cubic, flip, thre, block_flag, nhwc_heat, s);
        else
            st = launch_scan_nhwc_t(static_cast<const float *>(hmp.ptr), hmp.image_stride, hmp.pixel_stride,
                                    kp_flip_dev, n, n_total, c, h, w, scale, cubic, flip, thre, block_flag, nhwc_heat, s);
        OG_TRY(st);
        return launch_fused_t(static_cast<const float *>(nhwc_heat), (size_t)c * h * w, kp_flip_dev, n, n, c, h, w,
                              scale, cubic, false, thre, cand_count, cand_keys, block_flag, block_list, n_active,
                              sm_count, false, false, s, launches);
    }
    if (hmp.dtype == OG_DTYPE_BF16)
        return launch_fused_t(static_cast<const __nv_bfloat16 *>(hmp.ptr), hmp.image_stride, kp_flip_dev, n,
                              n_total, c, h, w, scale, cubic, flip, thre, cand_count, cand_keys, block_flag,
                              block_list, n_active, sm_count, clear_first, true, s, launches);
    if (hmp.dtype == OG_DTYPE_F16)
        return launch_fused_t(static_cast<const __half *>(hmp.ptr), hmp.image_stride, kp_flip_dev, n,
                              n_total, c, h, w, scale, cubic, flip, thre, cand_count, cand_keys, block_flag,
                              block_list, n_active, sm_count, clear_first, true, s, launches);
    return launch_fused_t(static_cast<const float *>(hmp.ptr), hmp.image_stride, kp_flip_dev, n, n_total, c,
                          h, w, scale, cubic, flip, thre, cand_count, cand_keys, block_flag, block_list,
                          n_active, sm_count, clear_first, true, s, launches);
}

// single network-resolution planes as dense float32, flip-fused (the exact per-plane redo of a
// fused decode: og_fetch_result resizes and radix-selects the planes whose candidate lists
// overflowed)
namespace {
template <typename T>
__global__ void fuse_planes_kernel(const T *__restrict__ hmp, size_t img_stride, size_t plane_stride,
                                   size_t pix_stride, const FlipTablesDev ft, int n,
                                   int C, int h, int w, int flip, const int32_t *__restrict__ plane_list,
                                   float *__restrict__ out) {
    const int plane = plane_list[blockIdx.y];
    const int img = plane / C, c = plane - img * C;
    const size_t hw = (size_t)h * w;
    const T *a = hmp + (size_t)img * img_stride + (size_t)c * plane_stride;
    const T *b = flip ? hmp + (size_t)(n + img) * img_stride + (size_t)ft.kp[c] * plane_stride : nullptr;
    float *o = out + (size_t)blockIdx.y * hw;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < hw; i += (size_t)gridDim.x * blockDim.x) {
        float v = load_cell(a + i * pix_stride);
        if (flip) {                          // (orig + flip_W(flipped)[kp_flip]) / 2, factory.py:101-106
            const int y = (int)(i / w), x = (int)(i - (size_t)y * w);
            v = __fmul_rn(__fadd_rn(v, load_cell(b + ((size_t)y * w + (w - 1 - x)) * pix_stride)), 0.5f);
        }
        o[i] = v;
    }
}
}  // namespace

int launch_fuse_planes(const MapView &hmp, const FlipTablesDev &flips, int n, int c, int h, int w, bool flip,
                       const int32_t *plane_list, int count, float *out, cudaStream_t s) {
    if (count == 0) return OG_OK;
    const size_t hw = (size_t)h * w;
    const dim3 grid((unsigned)std::min<size_t>((hw + 255) / 256, 64), (unsigned)count);
    if (hmp.dtype == OG_DTYPE_BF16)
        fuse_planes_kernel<<<grid, 256, 0, s>>>(static_cast<const __nv_bfloat16 *>(hmp.ptr), hmp.image_stride, hmp.plane_stride, hmp.pixel_stride, flips, n, c, h, w, flip ? 1 : 0, plane_list, out);
    else if (hmp.dtype == OG_DTYPE_F16)
        fuse_planes_kernel<<<grid, 256, 0, s>>>(static_cast<const __half *>(hmp.ptr), hmp.image_stride, hmp.plane_stride, hmp.pixel_stride, flips, n, c, h, w, flip ? 1 : 0, plane_list, out);
    else
        fuse_planes_kernel<<<grid, 256, 0, s>>>(static_cast<const float *>(hmp.ptr), hmp.image_stride, hmp.plane_stride, hmp.pixel_stride, flips, n, c, h, w, flip ? 1 : 0, plane_list, out);
    OG_CUDA_TRY(cudaGetLastError());
    return OG_OK;
}

}  // namespace og
