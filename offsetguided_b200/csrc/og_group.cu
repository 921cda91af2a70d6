// K3 — greedy limb-ordered keypoint grouping (reference decoder/group.py:39-240, which
// runs per image in a CPU process pool).  Three kernels:
//
//   prepare (og_prep.cuh)  one CTA per (limb type, image): the part of every limb step that
//       depends on the limb rows only — distance / border gate (group.py:64-76), sort by limb
//       score (canonical stable order) and "best row per to-joint id" (group.py:222-240).
//       All L x N instances run in parallel, off the sequential path.  On the decode path it
//       is the tail of K2's CTA (og_limbs.cu); group_prepare_kernel is the stand-alone form.
//   group_warp_kernel      ONE WARP per image walks the skeleton in the reference's limb order
//       over the compacted kept rows.  The walk is latency-bound (a few hundred pair tests per
//       limb type), so what counts is the length of the dependent chain: lane = person, every
//       person row is read and written by its own lane only, the cross-lane facts (how many
//       persons matched limb j, did any replacement pass) are warp votes, and the phases are
//       separated by __syncwarp instead of CTA barriers.  Loops are kept ROLLED: a lone warp
//       has nobody to hide instruction fetches behind, and the unrolled body (58 KB of SASS)
//       ran 5x slower than its dependent chain.  The person table is `warp_rows` rows
//       of shared memory (26 KB for 64 rows x 17 joints), so eight images share an SM.
//   group_kernel           one 256-thread CTA per image, table in the image's global slab of
//       L*K rows: the images whose table outgrew the warp kernel's (noise inputs), flagged by
//       it in `redo`; every other CTA of this launch exits at once.
//
// The person table (shared memory in the warp kernel, the slab in the CTA kernel) holds three
// planes per (person row, joint):
//   ids   int32   global keypoint id (-1 = unset)          pose column 5
//   score float   best limb score seen for the joint       pose column 4
//   xyvs  float4  x, y, keypoint score, keypoint scale     pose columns 0..3
// Persons are addressed through an `order` list (logical position -> table row), so
// deleting merged persons is a compaction of that small list, never a row move.
//
// The numpy program is sequential only in appearance; per limb type it is
//   (1) match every person against every kept limb   -> one thread per (person, limb) pair
//   (2) apply "both ends known" / "one end known"    -> one thread per person; the
//       reference's fancy-index scatter semantics (row-major pair order, last pair wins,
//       right-hand sides read before the statement) reduce to "the LAST kept limb that
//       matches person m" (atomicMax over the pair threads), applied by the thread owning m
//   (3) merge persons sharing exactly two ids        -> one thread per person pair; partner
//       = largest b (atomicMax); survivors read rows that are being deleted, which nobody
//       writes
//   (4) append unclaimed limbs as new persons, using the reference's column-sum rule
//       including its (-1)+(+1) cancellation quirk (group.py:166).
// The slab cannot overflow: every new person consumes one kept limb row, and there are at most
// L*K of those.
#include "og_common.cuh"
#include "og_prep.cuh"

#include <mutex>

namespace og {

namespace {

#ifndef OG_K3_THREADS
#define OG_K3_THREADS 256
#endif
constexpr int kGroupThreads = OG_K3_THREADS;
constexpr int kPrepThreads = 128;          // one thread per limb row, >= OG_MAX_TOPK
static_assert(kPrepThreads >= OG_MAX_TOPK, "prepare kernel needs one thread per limb row");

// Optional phase profile (build with -DOG_K3_PROFILE): thread 0 accumulates clock64()
// deltas per phase into og_k3_prof[phase]; og_k3_prof[15] counts CTAs.
#ifdef OG_K3_PROFILE
__device__ unsigned long long og_k3_prof[16];
#define OG_K3_PROF(ph)                                   \
    do {                                                 \
        if (threadIdx.x == 0) {                          \
            const long long t__ = clock64();             \
            prof_acc[ph] += t__ - prof_last;             \
            prof_last = t__;                             \
        }                                                \
    } while (0)
#else
#define OG_K3_PROF(ph) do { } while (0)
#endif

enum Flag { kAnyP1 = 0, kAnyP2, kAnyMerge, kOutOffset, kNNew, kNumFlags = 8 };

struct GroupArgs {
    int C, L, K;
    SkeletonDev sk;
    double person_thre;
    int sort_dim;
    int warp_rows;
    float *slab;     // per image: xyvs float4[PMAX*C], score float[PMAX*C], ids int[PMAX*C]
    size_t slab_stride;
    CocoOut coco;    // optional back-projected result rows (frames == nullptr: off)
    int32_t *lazy_flag;   // warp kernel: set when some image needs the CTA kernel (nullptr: it always follows)
};

// Result rows as the reference's evaluation loop builds them from the poses of one image
// (evaluate.py:227-265 after transforms/preprocess.py:33-63 annotations_inverse): per joint
// x, y moved back into the original image frame — (x + offset) / scale, each step evaluated in
// float64 and rounded to float32 like numpy's in-place updates of a float32 array — then
// np.around(., 2) in float32 (multiply by 100, rint, divide), and the flag "x > 0 or y > 0".
__device__ __forceinline__ void coco_joint(const double *__restrict__ frame, float x, float y,
                                           float *__restrict__ o) {
    const float x1 = __double2float_rn((double)x + frame[0]);
    const float y1 = __double2float_rn((double)y + frame[1]);
    const float x2 = __double2float_rn((double)x1 / frame[2]);
    const float y2 = __double2float_rn((double)y1 / frame[3]);
    const float x3 = __fdiv_rn(rintf(__fmul_rn(x2, 100.0f)), 100.0f);
    const float y3 = __fdiv_rn(rintf(__fmul_rn(y2, 100.0f)), 100.0f);
    o[0] = x3;
    o[1] = y3;
    o[2] = (x3 > 0.0f || y3 > 0.0f) ? 1.0f : 0.0f;
}

__host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---------------------------------------------------------------------------
// prepare, stand-alone (limb tables supplied by the caller; the decode path runs the same
// code at the end of K2): one CTA per (limb type, image)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kPrepThreads)
group_prepare_kernel(const float *__restrict__ limbs, int L, int K, float dist_max, int use_scale,
                     int32_t *__restrict__ prep, float4 *__restrict__ rec, int32_t *__restrict__ cnt) {
    __shared__ PrepShared<kPrepThreads> sh;
    const int tid = threadIdx.x;
    const size_t inst = (size_t)blockIdx.y * L + blockIdx.x;          // (image, limb type)
    float r[OG_LIMB_COLS];
#pragma unroll
    for (int i = 0; i < OG_LIMB_COLS; ++i) r[i] = 0.0f;
    if (tid < K) {
        const float *src = limbs + (inst * K + tid) * OG_LIMB_COLS;
#pragma unroll
        for (int i = 0; i < OG_LIMB_COLS; ++i) r[i] = __ldg(src + i);
    }
    prepare_limb_rows(r, tid, K, dist_max, use_scale, sh, prep + inst * (K + 1), rec + inst * K * 3,
                      cnt + inst);
}

// ---------------------------------------------------------------------------
// grouping
// ---------------------------------------------------------------------------
struct Layout {
    size_t conn, rows, k_int, p_i32, p_i16, p_u8, p_f64, warp, flags, total;
};

// k_int: 6 int arrays of K; p_i32: 3 int arrays of PMAX; p_i16: 3 int16 arrays of PMAX
__host__ __device__ inline Layout make_layout(int L, int K) {
    const size_t pmax = (size_t)L * K;
    Layout lo;
    size_t at = 0;
    lo.conn = at;  at += 2 * align_up((size_t)K * OG_LIMB_COLS * 4, 16);     // double buffer
    lo.rows = at;  at += 2 * align_up((size_t)(K + 1) * 4, 16);               // kept rows + count
    lo.k_int = at; at += (size_t)6 * K * 4;
    at = align_up(at, 8);
    lo.p_f64 = at; at += pmax * 8;
    lo.p_i32 = at; at += (size_t)3 * pmax * 4;
    lo.p_i16 = at; at += align_up((size_t)3 * pmax * 2, 4);
    lo.p_u8 = at;  at += align_up(pmax, 4);
    lo.warp = at;  at += 32 * 4;
    lo.flags = at; at += kNumFlags * 4;
    lo.total = align_up(at, 16);
    return lo;
}

// Exclusive scan of a predicate over [0, n): pos[i] = number of true entries before
// i (written for every i < n); returns the total.  All threads must call it.
template <typename Pred>
__device__ int block_scan(int n, Pred pred, int16_t *pos, int *s_warp) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int running = 0;
    for (int base = 0; base < n; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const bool f = (i < n) && pred(i);
        const unsigned ballot = __ballot_sync(0xffffffffu, f);
        if (lane == 0) s_warp[wid] = __popc(ballot);
        __syncthreads();
        int before = 0, tot = 0;
        for (int w = 0; w < nw; ++w) {
            const int c = s_warp[w];
            if (w < wid) before += c;
            tot += c;
        }
        if (i < n) pos[i] = (int16_t)(running + before + __popc(ballot & ((1u << lane) - 1u)));
        running += tot;
        __syncthreads();
    }
    return running;
}

// numpy's float32 pairwise summation for n <= 128 (loops_utils.h.src, probed).
__device__ float numpy_sum_f32(const float *a, int n) {
    if (n < 8) {
        float s = 0.0f;
        for (int i = 0; i < n; ++i) s = __fadd_rn(s, a[i]);
        return s;
    }
    float r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = a[j];
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = __fadd_rn(r[j], a[i + j]);
    }
    float s = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                        __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
    for (; i < n; ++i) s = __fadd_rn(s, a[i]);
    return s;
}

__device__ __forceinline__ float4 max4(float4 a, float4 b) {
    return make_float4(fmaxf(a.x, b.x), fmaxf(a.y, b.y), fmaxf(a.z, b.z), fmaxf(a.w, b.w));
}
__device__ __forceinline__ float unset_to_zero(float v) { return v == -1.0f ? 0.0f : v; }

__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gmem_src) {
    const unsigned saddr = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(saddr), "l"(gmem_src));
}

__global__ void __launch_bounds__(kGroupThreads)
group_kernel(GroupArgs a, const float *__restrict__ limbs, const int32_t *__restrict__ prep,
             float *__restrict__ out_poses, int capacity_rows, int32_t *__restrict__ out_offset,
             int32_t *__restrict__ out_count, int32_t *__restrict__ out_total,
             const int32_t *__restrict__ redo) {
    extern __shared__ __align__(16) unsigned char smem[];
    if (redo != nullptr && redo[blockIdx.x] == 0) return;       // the warp kernel finished this image
#ifdef OG_K3_PROFILE
    long long prof_acc[10] = {0};
    long long prof_last = clock64();
#endif
    const int C = a.C, L = a.L, K = a.K;
    const int pmax = L * K;
    const Layout lo = make_layout(L, K);
    const int tid = threadIdx.x, T = blockDim.x;
    const int lane = tid & 31, wid = tid >> 5;
    const int img = blockIdx.x;

    float *s_conn_buf[2];
    s_conn_buf[0] = reinterpret_cast<float *>(smem + lo.conn);
    s_conn_buf[1] = s_conn_buf[0] + align_up((size_t)K * OG_LIMB_COLS * 4, 16) / 4;
    int *s_rows_buf[2];                     // [0..K) kept rows in order, [K] their count
    s_rows_buf[0] = reinterpret_cast<int *>(smem + lo.rows);
    s_rows_buf[1] = s_rows_buf[0] + align_up((size_t)(K + 1) * 4, 16) / 4;
    int *kbase = reinterpret_cast<int *>(smem + lo.k_int);
    int *s_kind1 = kbase + 0 * K;
    int *s_kind2 = kbase + 1 * K;
    float *s_kscore = reinterpret_cast<float *>(kbase + 2 * K);
    int *s_n1 = kbase + 3 * K;
    int *s_n2 = kbase + 4 * K;
    int *s_new = kbase + 5 * K;
    int *p32 = reinterpret_cast<int *>(smem + lo.p_i32);
    int *s_pk1 = p32 + 0 * pmax;
    int *s_pk2 = p32 + 1 * pmax;
    int *s_blast = p32 + 2 * pmax;
    int16_t *pbase = reinterpret_cast<int16_t *>(smem + lo.p_i16);
    int16_t *s_order = pbase + 0 * pmax;
    int16_t *s_order2 = pbase + 1 * pmax;
    int16_t *s_pos = pbase + 2 * pmax;
    uint8_t *s_del = smem + lo.p_u8;
    double *s_ps = reinterpret_cast<double *>(smem + lo.p_f64);
    int *s_warp = reinterpret_cast<int *>(smem + lo.warp);
    volatile int *s_flag = reinterpret_cast<volatile int *>(smem + lo.flags);

    const float *limbs_img = limbs + (size_t)img * L * K * OG_LIMB_COLS;
    const int32_t *prep_img = prep + (size_t)img * L * (K + 1);

    float *slab_img = a.slab + (size_t)img * a.slab_stride;
    float4 *xyvs = reinterpret_cast<float4 *>(slab_img);
    float *score = slab_img + (size_t)pmax * C * 4;
    int *ids = reinterpret_cast<int *>(slab_img + (size_t)pmax * C * 5);
    int mm = 0, nalloc = 0;

    // rows and kept list of limb type li + 1 are fetched with cp.async while type li runs
    auto fetch_rows = [&](int li_next) {
        float *dst = s_conn_buf[li_next & 1];
        const float *src = limbs_img + (size_t)li_next * K * OG_LIMB_COLS;
        for (int i = tid; i < K * OG_LIMB_COLS; i += T) cp_async4(dst + i, src + i);
        int *rdst = s_rows_buf[li_next & 1];
        const int32_t *rsrc = prep_img + (size_t)li_next * (K + 1);
        for (int i = tid; i <= K; i += T) cp_async4(rdst + i, rsrc + i);
        asm volatile("cp.async.commit_group;");
    };
    fetch_rows(0);
    for (int li = 0; li < L; ++li) {
        const int jf = a.sk.from[li], jt = a.sk.to[li];
        const float *s_conn = s_conn_buf[li & 1];
        const int *s_rows = s_rows_buf[li & 1];
        asm volatile("cp.async.wait_all;" ::: "memory");        // data of type li has landed
        if (tid < kNumFlags) s_flag[tid] = 0;
        __syncthreads();
        // The buffers of type li + 1 are those of type li - 1: only after the barrier has every
        // thread finished reading them (a type with kk == 0 leaves its iteration without one).
        if (li + 1 < L) fetch_rows(li + 1);
        OG_K3_PROF(0);
        const int kk = s_rows[K];
        if (kk == 0) continue;                                         // group.py:84-85

        // ---- stage ids / scores of the kept rows; reset the per-person match slots
        for (int j = tid; j < kk; j += T) {
            const float *r = s_conn + s_rows[j] * OG_LIMB_COLS;
            s_kind1[j] = (int)r[6];
            s_kind2[j] = (int)r[7];
            s_kscore[j] = r[10];
            s_n1[j] = 0;
            s_n2[j] = 0;
        }
        for (int m = tid; m < mm; m += T) {
            s_pk1[m] = -1;
            s_pk2[m] = -1;
            s_blast[m] = -1;
            s_del[m] = 0;
        }
        __syncthreads();
        OG_K3_PROF(1);
        // ---- match persons x kept limbs on the pre-update snapshot (group.py:87-109),
        //      one thread per pair; the last matching limb of a person wins (atomicMax)
        for (int e = tid; e < mm * kk; e += T) {
            const int m = e / kk, j = e - m * kk;
            const int row = s_order[m];
            const int ms = (ids[row * C + jf] == s_kind1[j] ? 1 : 0) +
                           (ids[row * C + jt] == s_kind2[j] ? 1 : 0);
            if (ms == 0) continue;
            const float sc = s_kscore[j];
            const bool rep = (sc > score[row * C + jt]) || (sc > score[row * C + jf]);
            if (ms == 2) {
                atomicAdd(&s_n2[j], 1);
                if (rep) {
                    atomicMax(&s_pk2[m], j);
                    s_flag[kAnyP2] = 1;
                }
            } else {
                atomicAdd(&s_n1[j], 1);
                if (rep) {
                    atomicMax(&s_pk1[m], j);
                    s_flag[kAnyP1] = 1;
                }
            }
        }
        __syncthreads();
        OG_K3_PROF(2);
        // ---- apply: both ends known (group.py:114-119), then one end known (:124-135)
        for (int m = tid; m < mm; m += T) {
            const int row = s_order[m];
            const int k2 = s_pk2[m];
            if (k2 >= 0) {
                const float sc = s_kscore[k2];
                score[row * C + jf] = fmaxf(sc, score[row * C + jf]);
                score[row * C + jt] = fmaxf(sc, score[row * C + jt]);
            }
            const int k1 = s_pk1[m];
            if (k1 >= 0) {
                const float *r = s_conn + s_rows[k1] * OG_LIMB_COLS;
                ids[row * C + jf] = s_kind1[k1];
                ids[row * C + jt] = s_kind2[k1];
                xyvs[row * C + jf] = make_float4(r[0], r[1], r[2], r[11]);
                xyvs[row * C + jt] = make_float4(r[3], r[4], r[5], r[12]);
                const float sc = s_kscore[k1];
                score[row * C + jf] = fmaxf(sc, score[row * C + jf]);
                score[row * C + jt] = fmaxf(sc, score[row * C + jt]);
            }
        }
        __syncthreads();
        OG_K3_PROF(3);
        // ---- merge persons sharing exactly two keypoint ids (group.py:140-155), one thread
        //      per ordered pair p < q; the largest partner of p wins
        int mm_after = mm;
        if (mm >= 2) {
            for (int e = tid; e < mm * mm; e += T) {
                const int p = e / mm, q = e - p * mm;
                if (q <= p) continue;
                const int rowa = s_order[p], rowb = s_order[q];
                int cnt = 0;
                for (int c = 0; c < C; ++c) {
                    const int ia = ids[rowa * C + c];
                    cnt += (ia != -1 && ia == ids[rowb * C + c]) ? 1 : 0;
                }
                if (cnt == 2) {
                    atomicMax(&s_blast[p], q);
                    s_del[q] = 1;
                    s_flag[kAnyMerge] = 1;
                }
            }
            __syncthreads();
            OG_K3_PROF(4);
            if (s_flag[kAnyMerge]) {
                for (int p = tid; p < mm; p += T) {
                    const int q = s_blast[p];
                    if (q < 0 || s_del[p]) continue;      // deleted rows are never read again
                    const int rowa = s_order[p], rowb = s_order[q];
                    for (int c = 0; c < C; ++c) {
                        ids[rowa * C + c] = max(ids[rowa * C + c], ids[rowb * C + c]);
                        score[rowa * C + c] = fmaxf(score[rowa * C + c], score[rowb * C + c]);
                        xyvs[rowa * C + c] = max4(xyvs[rowa * C + c], xyvs[rowb * C + c]);
                    }
                }
                mm_after = block_scan(mm, [&](int p) { return s_del[p] == 0; }, s_pos, s_warp);
                for (int p = tid; p < mm; p += T)
                    if (!s_del[p]) s_order2[s_pos[p]] = s_order[p];
                __syncthreads();
                int16_t *tmp = s_order;
                s_order = s_order2;
                s_order2 = tmp;
            }
        }
        // ---- warp 0: unclaimed limbs start new persons (group.py:166-177), column-sum
        //      rule with its (-1) + (+1) cancellation
        if (wid == 0) {
            const int w2 = s_flag[kAnyP2] ? -1 : 2;
            const int w1 = s_flag[kAnyP1] ? -1 : 1;
            int nnew = 0;
            for (int j0 = 0; j0 < kk; j0 += 32) {
                const int j = j0 + lane;
                const bool isnew = j < kk && (s_n2[j] * w2 + s_n1[j] * w1 == 0);
                const unsigned mask = __ballot_sync(0xffffffffu, isnew);
                if (isnew) s_new[nnew + __popc(mask & ((1u << lane) - 1u))] = j;
                nnew += __popc(mask);
            }
            if (lane == 0) s_flag[kNNew] = nnew;
        }
        __syncthreads();
        OG_K3_PROF(5);
        const int nnew = s_flag[kNNew];
        for (int e = tid; e < nnew * C; e += T) {
            const int q = e / C, c = e - q * C;
            const int j = s_new[q];
            const int at = (nalloc + q) * C + c;
            const float *r = s_conn + s_rows[j] * OG_LIMB_COLS;
            if (c == 0) s_order[mm_after + q] = (int16_t)(nalloc + q);
            if (c == jt) {
                ids[at] = s_kind2[j];
                xyvs[at] = make_float4(r[3], r[4], r[5], r[12]);
                score[at] = s_kscore[j];
            } else if (c == jf) {
                ids[at] = s_kind1[j];
                xyvs[at] = make_float4(r[0], r[1], r[2], r[11]);
                score[at] = s_kscore[j];
            } else {
                ids[at] = -1;
                xyvs[at] = make_float4(-1.f, -1.f, -1.f, -1.f);
                score[at] = -1.0f;
            }
        }
        nalloc += nnew;
        mm = mm_after + nnew;
        __syncthreads();
        OG_K3_PROF(6);
    }
    asm volatile("cp.async.wait_all;" ::: "memory");

    // ---- person score, threshold, stable descending sort (group.py:188-219)
    for (int m = tid; m < mm; m += T) {
        const int row = s_order[m];
        float vals[OG_MAX_KEYPOINTS];
        int n = 0;
        for (int c = 0; c < C; ++c) {
            float v;
            const float4 q = xyvs[row * C + c];
            switch (a.sort_dim) {
                case 0: v = q.x; break;
                case 1: v = q.y; break;
                case 2: v = q.z; break;
                case 3: v = q.w; break;
                case 4: v = score[row * C + c]; break;
                default: v = (float)ids[row * C + c]; break;
            }
            if (v > 0.0f) vals[n++] = v;
        }
        const double ps = (double)numpy_sum_f32(vals, n) / (double)n;      // 0/0 -> NaN, kept
        s_ps[m] = ps;
        s_del[m] = (ps < a.person_thre) ? 1 : 0;
    }
    __syncthreads();
    const int nk = block_scan(mm, [&](int m) { return s_del[m] == 0; }, s_pos, s_warp);
    for (int m = tid; m < mm; m += T)
        if (!s_del[m]) s_order2[s_pos[m]] = (int16_t)m;        // kept persons, original order
    __syncthreads();
    for (int q = tid; q < nk; q += T) {
        double ps = s_ps[s_order2[q]];
        if (ps != ps) ps = -1.0e300;        // documented deviation: NaN scores sort last
        int rank = 0;
        for (int q2 = 0; q2 < nk; ++q2) {
            double p2 = s_ps[s_order2[q2]];
            if (p2 != p2) p2 = -1.0e300;
            rank += (p2 > ps || (p2 == ps && q2 < q)) ? 1 : 0;
        }
        s_blast[q] = rank;
    }
    if (tid == 0) {
        const int off = atomicAdd(out_total, nk);
        s_flag[kOutOffset] = off;
        out_offset[img] = off;
        out_count[img] = nk;
    }
    __syncthreads();
    OG_K3_PROF(7);
    const int off = s_flag[kOutOffset];
    for (int e = tid; e < nk * C; e += T) {
        const int q = e / C, c = e - q * C;
        const int dst = off + s_blast[q];
        if (dst >= capacity_rows) continue;
        const int row = s_order[s_order2[q]];
        const float4 v = xyvs[row * C + c];
        float *o = out_poses + ((size_t)dst * C + c) * OG_POSE_COLS;
        o[0] = unset_to_zero(v.x);
        o[1] = unset_to_zero(v.y);
        o[2] = unset_to_zero(v.z);
        o[3] = unset_to_zero(v.w);
        o[4] = unset_to_zero(score[row * C + c]);
        o[5] = unset_to_zero((float)ids[row * C + c]);
        if (a.coco.frames != nullptr) {
            coco_joint(a.coco.frames + (size_t)(a.coco.image0 + img) * 4, unset_to_zero(v.x), unset_to_zero(v.y),
                       a.coco.keypoints + ((size_t)dst * C + c) * 3);
            if (c == 0) {       // score = sum(v) / len(v), float64, left to right (evaluate.py:250)
                double acc = 0.0;
                for (int cc = 0; cc < C; ++cc) acc += (double)unset_to_zero(xyvs[row * C + cc].z);
                a.coco.scores[dst] = acc / (double)C;
                a.coco.images[dst] = a.coco.image0 + img;
            }
        }
    }
#ifdef OG_K3_PROFILE
    OG_K3_PROF(8);
    if (threadIdx.x == 0) {
        for (int ph = 0; ph < 10; ++ph) atomicAdd(&og_k3_prof[ph], (unsigned long long)prof_acc[ph]);
        atomicAdd(&og_k3_prof[15], 1ull);
    }
#endif
}

// ---------------------------------------------------------------------------
// grouping, one warp per image
// ---------------------------------------------------------------------------
struct WarpLayout {
    size_t xyvs, score, ids, rec, k_int, p_f64, p_i32, p_i16, p_u8, cnt, total;
};

// Kept rows are fetched kRecRing - 1 limb types ahead: a limb step of the register path is ~1000
// cycles, less than one L2 round trip of the rows behind it.
constexpr int kRecRing = 4;

// Person-table rows are CS entries apart, CS = the multiple of 4 >= C with CS % 8 == 4: a row of
// ids is a few aligned 128-bit words (the pair test of the merge step compares whole rows), the
// quarter-warps of such loads hit distinct banks, and column accesses of 32 different rows
// conflict at most 4-way.  Pad columns hold "unset".
__host__ __device__ inline int warp_row_stride(int C) {
    int cs = (C + 3) / 4 * 4;
    if (cs % 8 == 0) cs += 4;
    return cs;
}

__host__ __device__ inline WarpLayout make_warp_layout(int C, int L, int K, int rows) {
    const size_t cs = (size_t)warp_row_stride(C);
    WarpLayout lo;
    size_t at = 0;
    lo.xyvs = at;  at += (size_t)rows * cs * 16;
    lo.score = at; at += (size_t)rows * cs * 4;
    lo.ids = at;   at += (size_t)rows * cs * 4;
    at = align_up(at, 16);
    lo.rec = at;   at += kRecRing * (size_t)K * 48;     // kept rows of the next limb types (prefetch ring)
    lo.k_int = at; at += (size_t)3 * K * 4;             // per kept row: persons matched at one / both ends, new list
    at = align_up(at, 8);
    lo.p_f64 = at; at += (size_t)rows * 8;              // person scores
    lo.p_i32 = at; at += (size_t)2 * rows * 4;          // merge partner / kept list, rank
    lo.p_i16 = at; at += align_up((size_t)rows * 2, 4); // order: logical position -> table row
    lo.p_u8 = at;  at += align_up((size_t)rows, 4);     // deleted marks
    lo.cnt = at;   at += (size_t)L * 4;
    lo.total = align_up(at, 16);
    return lo;
}

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    const unsigned saddr = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(gmem_src));
}

// e / d for 0 <= e < 65536, 1 <= d <= 256 without an integer division: (e + 0.5) / d lies at
// least 0.5 / d away from an integer, far more than the error of the approximate reciprocal
__device__ __forceinline__ int small_div(int e, float inv_d) {
    return __float2int_rz(((float)e + 0.5f) * inv_d);
}

__global__ void __launch_bounds__(32)
group_warp_kernel(GroupArgs a, const float4 *__restrict__ rec, const int32_t *__restrict__ cnt,
                  float *__restrict__ out_poses, int capacity_rows, int32_t *__restrict__ out_offset,
                  int32_t *__restrict__ out_count, int32_t *__restrict__ out_total,
                  int32_t *__restrict__ redo) {
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr unsigned kAll = 0xffffffffu;
    const int C = a.C, L = a.L, K = a.K, R = a.warp_rows;
    const int CS = warp_row_stride(C), NV = CS / 4;
    const WarpLayout lo = make_warp_layout(C, L, K, R);
#ifdef OG_K3_PROFILE
    long long prof_acc[10] = {0};
    long long prof_last = clock64();
#endif
    const int lane = threadIdx.x;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int img = blockIdx.x;

    // every pointer below is derived from `smem` by plain arithmetic, so the accesses compile to
    // LDS / STS (a pointer picked out of an array of pointers degrades to generic loads)
    float4 *xyvs = reinterpret_cast<float4 *>(smem + lo.xyvs);
    float *score = reinterpret_cast<float *>(smem + lo.score);
    int *ids = reinterpret_cast<int *>(smem + lo.ids);
    float4 *s_rec0 = reinterpret_cast<float4 *>(smem + lo.rec);
    int *s_n1 = reinterpret_cast<int *>(smem + lo.k_int);
    int *s_n2 = s_n1 + K;
    int *s_new = s_n2 + K;
    double *s_ps = reinterpret_cast<double *>(smem + lo.p_f64);
    int *s_pa = reinterpret_cast<int *>(smem + lo.p_i32);     // per person: winning limb (one end known) / merge partner / kept list
    int *s_pb = s_pa + R;                                     // per person: winning limb (both ends known) / rank
    int16_t *s_order = reinterpret_cast<int16_t *>(smem + lo.p_i16);
    uint8_t *s_del = smem + lo.p_u8;
    int *s_cnt = reinterpret_cast<int *>(smem + lo.cnt);

    const float4 *rec_img = rec + (size_t)img * L * K * 3;
#pragma unroll 1
    for (int l = lane; l < L; l += 32) s_cnt[l] = __ldg(cnt + (size_t)img * L + l);
    __syncwarp();

    // the kept rows of limb types li + 1 .. li + kRecRing - 1 arrive (cp.async) while type li is
    // processed; every call commits one group (an empty one past the last type), so "at most
    // kRecRing - 2 groups pending" always means "type li has landed"
    auto fetch_rows = [&](int li) {
        if (li < L) {
            const int n16 = (s_cnt[li] & kPrepCountMask) * 3;
            float4 *dst = s_rec0 + (size_t)(li % kRecRing) * K * 3;
            const float4 *src = rec_img + (size_t)li * K * 3;
#pragma unroll 1
            for (int i = lane; i < n16; i += 32) cp_async16(dst + i, src + i);
        }
        asm volatile("cp.async.commit_group;");
    };
#pragma unroll 1
    for (int li = 0; li < kRecRing - 1; ++li) fetch_rows(li);

    int mm = 0, nalloc = 0;
    // `dirty`: some pair of persons may share exactly two ids although no id changes in this step
    // (a merge or a "cancellation" person of an earlier step); see the merge step below
    bool dirty = false;
#pragma unroll 1
    for (int li = 0; li < L; ++li) {
        const int kk = s_cnt[li] & kPrepCountMask;
        const bool dup_from = (s_cnt[li] & kPrepDupFrom) != 0;     // two kept rows start at the same joint id
        asm volatile("cp.async.wait_group %0;" ::"n"(kRecRing - 2) : "memory");
        __syncwarp();          // rows of type li have landed; everybody is done with type li - 1
        fetch_rows(li + kRecRing - 1);
        OG_K3_PROF(0);
        if (kk == 0) continue;                                             // group.py:84-85
        const int jf = a.sk.from[li], jt = a.sk.to[li];
        const float4 *s_rec = s_rec0 + (size_t)(li % kRecRing) * K * 3;
        if (mm <= 32 && kk <= 32) {
            // ================= register path: at most 32 persons and 32 kept rows ==============
            // lane = person AND lane = kept row.  The limb step is a chain of dependent steps, so
            // what it costs is the length of that chain: here the table is touched twice (the
            // person's two joints before the match, its id row before the merge test) and all
            // cross-lane traffic is shuffles, votes and MATCH instead of shared-memory atomics.
            float4 r0 = make_float4(0.f, 0.f, 0.f, 0.f), r1 = r0, r2 = r0;
            if (lane < kk) {
                r0 = s_rec[lane * 3];
                r1 = s_rec[lane * 3 + 1];
                r2 = s_rec[lane * 3 + 2];
            }
            const int my_id1 = __float_as_int(r0.x), my_id2 = __float_as_int(r0.y);
            const bool live = lane < mm;
            const int my_ord = live ? (int)s_order[lane] : 0;
            const int row = my_ord * CS;
            const int at_f = row + jf, at_t = row + jt;
            int id_f = 0, id_t = 0;
            float sc_f = 0.f, sc_t = 0.f;
            if (live) {
                id_f = ids[at_f];
                id_t = ids[at_t];
                sc_f = score[at_f];
                sc_t = score[at_t];
            }
            // ---- match (group.py:87-109): every lane walks the kept rows (one broadcast 128-bit
            //      load each, no cross-lane traffic inside the loop) and collects three bit sets over
            //      them: rows that start / end at this person's joint ids, rows whose score passes
            //      the replacement test.  m1 / m2: rows matched at one end / at both ends; the LAST
            //      replacing row of each kind wins (row-major fancy-index scatter).
            unsigned mf = 0u, mt = 0u, mrep = 0u;
            const float sc_min = fminf(sc_t, sc_f);         // sc > sc_t || sc > sc_f (fminf drops a NaN like the two tests do)
#pragma unroll 4
            for (int j = 0; j < kk; ++j) {
                const float4 q = s_rec[j * 3];
                const unsigned bit = 1u << j;
                if (id_f == __float_as_int(q.x)) mf |= bit;
                if (id_t == __float_as_int(q.y)) mt |= bit;
                if (q.z > sc_min) mrep |= bit;
            }
            if (!live) mf = mt = 0u;
            const unsigned m2 = mf & mt, m1 = mf ^ mt;
            const int pk2 = 31 - __clz(m2 & mrep), pk1 = 31 - __clz(m1 & mrep);      // -1: none
            int pk1_i1 = 0, pk1_i2 = 0;
            float pk1_sc = 0.f, pk2_sc = 0.f;
            if (pk1 >= 0) {
                const float4 q = s_rec[pk1 * 3];
                pk1_i1 = __float_as_int(q.x);
                pk1_i2 = __float_as_int(q.y);
                pk1_sc = q.z;
            }
            if (pk2 >= 0) pk2_sc = s_rec[pk2 * 3].z;
            const unsigned any1 = __reduce_or_sync(kAll, m1), any2 = __reduce_or_sync(kAll, m2);
            const unsigned matched = any1 | any2;           // kept rows some person matches
            const bool any_p2 = __any_sync(kAll, pk2 >= 0), any_p1 = __any_sync(kAll, pk1 >= 0);
            // ---- does the merge step have anything to find?  (group.py:140-155 compares every pair
            //      of persons over all joints in every step.)  A pair's number of shared ids only
            //      changes when a "one end known" update rewrites a joint id, and then only
            //        - downwards, if the rewritten slot held an id before            (`lost`), or
            //        - upwards, if two persons end up holding the same id of this limb type: both
            //          match the same kept row (`overlap`), or their rows start at the same joint
            //          (`dup_from`).
            //      Without any of these — the normal step: unset joints filled in — no pair count
            //      changes, and a table without a pair sharing exactly two ids (`!dirty`) stays so.
            bool need_scan = dirty;
            if (!need_scan && any_p1) {
                const bool lost = pk1 >= 0 && ((id_t != pk1_i2 && id_t != -1) || (id_f != pk1_i1 && id_f != -1));
                const bool overlap = __reduce_add_sync(kAll, (unsigned)__popc(m1 | m2)) > (unsigned)__popc(matched);
                need_scan = overlap || dup_from || __any_sync(kAll, lost);
            }
            OG_K3_PROF(1);
            // ---- apply (group.py:114-135): both ends known, then one end known
            if (pk2 >= 0) {
                sc_f = fmaxf(pk2_sc, sc_f);
                sc_t = fmaxf(pk2_sc, sc_t);
            }
            if (pk1 >= 0) {
                ids[at_f] = pk1_i1;
                ids[at_t] = pk1_i2;
                xyvs[at_f] = s_rec[pk1 * 3 + 1];
                xyvs[at_t] = s_rec[pk1 * 3 + 2];
                sc_f = fmaxf(pk1_sc, sc_f);
                sc_t = fmaxf(pk1_sc, sc_t);
            }
            if (pk1 >= 0 || pk2 >= 0) {
                score[at_f] = sc_f;
                score[at_t] = sc_t;
            }
            __syncwarp();
            OG_K3_PROF(2);
            // ---- merge (group.py:140-155).  Per joint column, MATCH gives every lane the set of
            //      persons holding the same keypoint id; bit-sliced counters add these sets up over
            //      the columns, and the persons sharing EXACTLY two ids fall out as one mask per lane.
            int mm_after = mm;
            if (mm >= 2 && need_scan) {
                dirty = false;
                unsigned ones = 0u, twos = 0u, fours = 0u, over = 0u;
                auto add_column = [&](int v) {
                    unsigned m = __match_any_sync(kAll, v);
                    m = (v == -1) ? 0u : (m & ~(1u << lane));
                    const unsigned c0 = ones & m;
                    ones ^= m;
                    const unsigned c1 = twos & c0;
                    twos ^= c0;
                    over |= fours & c1;
                    fours ^= c1;
                };
                if (NV == 5) {
                    int4 x[5];
#pragma unroll
                    for (int v = 0; v < 5; ++v)
                        x[v] = live ? reinterpret_cast<const int4 *>(ids + row)[v] : make_int4(-1, -1, -1, -1);
#pragma unroll
                    for (int v = 0; v < 5; ++v) {
                        add_column(x[v].x);
                        add_column(x[v].y);
                        add_column(x[v].z);
                        add_column(x[v].w);
                    }
                } else {
#pragma unroll 1
                    for (int c = 0; c < C; ++c) add_column(live ? ids[row + c] : -1);
                }
                const unsigned two_shared = twos & ~ones & ~fours & ~over;
                OG_K3_PROF(4);
                if (__any_sync(kAll, two_shared != 0u)) {
                    // the relation is symmetric: q is deleted iff it shares two ids with a smaller p;
                    // a surviving p takes the element-wise maximum with its LARGEST partner
                    const bool del = (two_shared & lt_mask) != 0u;
                    const int partner = two_shared ? 31 - __clz(two_shared) : -1;
                    if (live && !del && partner > lane) {
                        const int rb = (int)s_order[partner] * CS;
#pragma unroll 1
                        for (int c = 0; c < C; ++c) {
                            ids[row + c] = max(ids[row + c], ids[rb + c]);
                            score[row + c] = fmaxf(score[row + c], score[rb + c]);
                            xyvs[row + c] = max4(xyvs[row + c], xyvs[rb + c]);
                        }
                    }
                    const bool keep = live && !del;
                    const unsigned kb = __ballot_sync(kAll, keep);
                    __syncwarp();
                    if (keep) s_order[__popc(kb & lt_mask)] = (int16_t)my_ord;
                    mm_after = __popc(kb);
                    dirty = true;           // merged rows may share two ids with a third person
                }
            }
            OG_K3_PROF(5);
            // ---- new persons (group.py:166-177), lane = kept row: column sum n2 * w2 + n1 * w1 == 0.
            //      With both weights of one sign this is "nobody matches the row"; with opposite
            //      signs a row matched at one end by as many persons as the weights balance
            //      cancels to 0 as well (the reference's quirk) — counted only for such rows.
            const int w2 = any_p2 ? -1 : 2, w1 = any_p1 ? -1 : 1;
            bool isnew = lane < kk && ((matched >> lane) & 1u) == 0u;
            if (any_p1 != any_p2) {
                unsigned both = any1 & any2;
#pragma unroll 1
                while (both) {
                    const int j = __ffs(both) - 1;
                    both &= both - 1u;
                    const int n2 = __popc(__ballot_sync(kAll, (m2 >> j) & 1u));
                    const int n1 = __popc(__ballot_sync(kAll, (m1 >> j) & 1u));
                    if (lane == j) isnew = (n2 * w2 + n1 * w1 == 0);
                }
            }
            // a person made from a row that somebody matches shares ids with that somebody
            if (__any_sync(kAll, isnew && ((matched >> lane) & 1u))) dirty = true;
            const unsigned nb = __ballot_sync(kAll, isnew);
            const int nnew = __popc(nb);
            if (nalloc + nnew > R) {
                asm volatile("cp.async.wait_all;" ::: "memory");
                if (lane == 0) {
                    redo[img] = 1;
                    if (a.lazy_flag) *a.lazy_flag = 1;
                }
                return;
            }
            if (isnew) {
                const int q = __popc(nb & lt_mask);
                const int base = (nalloc + q) * CS;
                const int4 unset_i = make_int4(-1, -1, -1, -1);
                const float4 unset_f = make_float4(-1.f, -1.f, -1.f, -1.f);
#pragma unroll 1
                for (int v = 0; v < NV; ++v) {
                    reinterpret_cast<int4 *>(ids + base)[v] = unset_i;
                    reinterpret_cast<float4 *>(score + base)[v] = unset_f;
                }
#pragma unroll 4
                for (int c = 0; c < CS; ++c) xyvs[base + c] = unset_f;          // CS is a multiple of 4
                ids[base + jf] = my_id1;
                ids[base + jt] = my_id2;
                score[base + jf] = r0.z;
                score[base + jt] = r0.z;
                xyvs[base + jf] = r1;
                xyvs[base + jt] = r2;
                s_order[mm_after + q] = (int16_t)(nalloc + q);
            }
            nalloc += nnew;
            mm = mm_after + nnew;
            OG_K3_PROF(6);
            continue;
        }
        // ================= general path: any table size, shared-memory work arrays =============
#pragma unroll 1
        for (int j = lane; j < kk; j += 32) {
            s_n1[j] = 0;
            s_n2[j] = 0;
        }
#pragma unroll 1
        for (int m = lane; m < mm; m += 32) {
            s_pa[m] = -1;
            s_pb[m] = -1;
        }
        __syncwarp();

        // ---- match persons x kept limbs on the pre-update table (group.py:87-109), one lane per
        //      pair: of the limbs that match a person the LAST one wins (fancy-index scatter in
        //      row-major pair order = atomicMax over the pair lanes)
        {
            const float inv_kk = __frcp_rn((float)kk);
#pragma unroll 1
            for (int e = lane; e < mm * kk; e += 32) {
                const int m = small_div(e, inv_kk), j = e - m * kk;
                const int row = (int)s_order[m] * CS;
                const float4 r0 = s_rec[j * 3];
                const int ms = (ids[row + jf] == __float_as_int(r0.x) ? 1 : 0) +
                               (ids[row + jt] == __float_as_int(r0.y) ? 1 : 0);
                if (ms == 0) continue;
                const bool rep = (r0.z > score[row + jt]) || (r0.z > score[row + jf]);
                if (ms == 2) {
                    atomicAdd(&s_n2[j], 1);
                    if (rep) atomicMax(&s_pb[m], j);
                } else {
                    atomicAdd(&s_n1[j], 1);
                    if (rep) atomicMax(&s_pa[m], j);
                }
            }
        }
        __syncwarp();
        OG_K3_PROF(1);
        // ---- apply, lane = person: both ends known (group.py:114-119), then one end known
        //      (:124-135); the slots are re-armed for the merge step on the way
        bool any_p1 = false, any_p2 = false;
#pragma unroll 1
        for (int mb = 0; mb < mm; mb += 32) {
            const int m = mb + lane;
            int pk1 = -1, pk2 = -1;
            if (m < mm) {
                pk1 = s_pa[m];
                pk2 = s_pb[m];
                s_pa[m] = -1;
                s_del[m] = 0;
                const int row = (int)s_order[m] * CS;
                const int at_f = row + jf, at_t = row + jt;
                if (pk2 >= 0) {
                    const float sc = s_rec[pk2 * 3].z;
                    score[at_f] = fmaxf(sc, score[at_f]);
                    score[at_t] = fmaxf(sc, score[at_t]);
                }
                if (pk1 >= 0) {
                    const float4 r0 = s_rec[pk1 * 3];
                    ids[at_f] = __float_as_int(r0.x);
                    ids[at_t] = __float_as_int(r0.y);
                    xyvs[at_f] = s_rec[pk1 * 3 + 1];
                    xyvs[at_t] = s_rec[pk1 * 3 + 2];
                    score[at_f] = fmaxf(r0.z, score[at_f]);
                    score[at_t] = fmaxf(r0.z, score[at_t]);
                }
            }
            any_p2 = any_p2 || __any_sync(kAll, pk2 >= 0);
            any_p1 = any_p1 || __any_sync(kAll, pk1 >= 0);
        }
        __syncwarp();
        OG_K3_PROF(2);

        // ---- merge persons sharing exactly two keypoint ids (group.py:140-155), one lane per
        //      pair p < q (pair e = q (q - 1) / 2 + p); the largest partner of p wins
        int mm_after = mm;
        if (mm >= 2) {
            bool found = false;
            const int npairs = mm * (mm - 1) / 2;
#pragma unroll 1
            for (int e = lane; e < npairs; e += 32) {
                int q = __float2int_rz((__fsqrt_rn(8.0f * (float)e + 1.0f) + 1.0f) * 0.5f);
                if (q * (q - 1) / 2 > e) --q;
                else if ((q + 1) * q / 2 <= e) ++q;
                const int p = e - q * (q - 1) / 2;
                const int4 *ia = reinterpret_cast<const int4 *>(ids + (int)s_order[p] * CS);
                const int4 *ib = reinterpret_cast<const int4 *>(ids + (int)s_order[q] * CS);
                int shared_ids = 0;
                auto count4 = [&](const int4 &x, const int4 &y) {
                    shared_ids += ((x.x != -1 && x.x == y.x) ? 1 : 0) + ((x.y != -1 && x.y == y.y) ? 1 : 0) +
                                  ((x.z != -1 && x.z == y.z) ? 1 : 0) + ((x.w != -1 && x.w == y.w) ? 1 : 0);
                };
                if (NV == 5) {                      // 17 (COCO) and 14 (CrowdPose) keypoints: ten loads in flight
                    int4 x[5], y[5];
#pragma unroll
                    for (int v = 0; v < 5; ++v) {
                        x[v] = ia[v];
                        y[v] = ib[v];
                    }
#pragma unroll
                    for (int v = 0; v < 5; ++v) count4(x[v], y[v]);
                } else {
#pragma unroll 1
                    for (int v = 0; v < NV; ++v) count4(ia[v], ib[v]);
                }
                if (shared_ids == 2) {
                    atomicMax(&s_pa[p], q);
                    s_del[q] = 1;
                    found = true;
                }
            }
            __syncwarp();
            OG_K3_PROF(4);
            if (__any_sync(kAll, found)) {
#pragma unroll 1
                for (int p = lane; p < mm; p += 32) {
                    const int q = s_pa[p];
                    if (q < 0 || s_del[p]) continue;          // deleted rows are never read again
                    const int ra = (int)s_order[p] * CS, rb = (int)s_order[q] * CS;
#pragma unroll 1
                    for (int c = 0; c < C; ++c) {
                        ids[ra + c] = max(ids[ra + c], ids[rb + c]);
                        score[ra + c] = fmaxf(score[ra + c], score[rb + c]);
                        xyvs[ra + c] = max4(xyvs[ra + c], xyvs[rb + c]);
                    }
                }
                __syncwarp();
                int kept = 0;                                  // compact the order list in place
#pragma unroll 1
                for (int mb = 0; mb < mm; mb += 32) {
                    const int m = mb + lane;
                    const bool keep = m < mm && s_del[m] == 0;
                    const int16_t row = keep ? s_order[m] : (int16_t)0;
                    const unsigned ballot = __ballot_sync(kAll, keep);
                    __syncwarp();
                    if (keep) s_order[kept + __popc(ballot & lt_mask)] = row;
                    kept += __popc(ballot);
                }
                mm_after = kept;
                __syncwarp();
            }
        }
        OG_K3_PROF(5);
        // ---- unclaimed limbs start new persons (group.py:166-177): column-sum rule with its
        //      (-1) + (+1) cancellation
        const int w2 = any_p2 ? -1 : 2, w1 = any_p1 ? -1 : 1;
        int nnew = 0;
#pragma unroll 1
        for (int j0 = 0; j0 < kk; j0 += 32) {
            const int j = j0 + lane;
            const bool isnew = j < kk && (s_n2[j] * w2 + s_n1[j] * w1 == 0);
            const unsigned ballot = __ballot_sync(kAll, isnew);
            if (isnew) s_new[nnew + __popc(ballot & lt_mask)] = j;
            nnew += __popc(ballot);
        }
        if (nalloc + nnew > R) {            // warp-uniform: the CTA kernel redoes this image
            asm volatile("cp.async.wait_all;" ::: "memory");
            if (lane == 0) {
                redo[img] = 1;
                if (a.lazy_flag) *a.lazy_flag = 1;
            }
            return;
        }
        if (nnew > 0) {
            __syncwarp();
            const float inv_cs = __frcp_rn((float)CS);
#pragma unroll 1
            for (int e = lane; e < nnew * CS; e += 32) {        // one lane per (new person, column); pad columns stay "unset"
                const int q = small_div(e, inv_cs), c = e - q * CS;
                const int j = s_new[q];
                const int at = (nalloc + q) * CS + c;
                if (c == jt) {
                    const float4 r0 = s_rec[j * 3];
                    ids[at] = __float_as_int(r0.y);
                    xyvs[at] = s_rec[j * 3 + 2];
                    score[at] = r0.z;
                } else if (c == jf) {
                    const float4 r0 = s_rec[j * 3];
                    ids[at] = __float_as_int(r0.x);
                    xyvs[at] = s_rec[j * 3 + 1];
                    score[at] = r0.z;
                } else {
                    ids[at] = -1;
                    xyvs[at] = make_float4(-1.f, -1.f, -1.f, -1.f);
                    score[at] = -1.0f;
                }
                if (c == 0) s_order[mm_after + q] = (int16_t)(nalloc + q);
            }
        }
        nalloc += nnew;
        mm = mm_after + nnew;
        dirty = true;           // the general path keeps no account of what it changed
        OG_K3_PROF(6);
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncwarp();

    // ---- person score, threshold, stable descending sort (group.py:188-219)
#pragma unroll 1
    for (int m = lane; m < mm; m += 32) {
        const int row = (int)s_order[m] * CS;
        float vals[OG_MAX_KEYPOINTS];
        int n = 0;
#pragma unroll 1
        for (int c = 0; c < C; ++c) {
            float v;
            const float4 q = xyvs[row + c];
            switch (a.sort_dim) {
                case 0: v = q.x; break;
                case 1: v = q.y; break;
                case 2: v = q.z; break;
                case 3: v = q.w; break;
                case 4: v = score[row + c]; break;
                default: v = (float)ids[row + c]; break;
            }
            if (v > 0.0f) vals[n++] = v;
        }
        const double ps = (double)numpy_sum_f32(vals, n) / (double)n;      // 0/0 -> NaN, kept
        s_ps[m] = ps;
        s_del[m] = (ps < a.person_thre) ? 1 : 0;
    }
    __syncwarp();
    int nk = 0;                                     // s_pa: kept persons in their original order
#pragma unroll 1
    for (int mb = 0; mb < mm; mb += 32) {
        const int m = mb + lane;
        const bool keep = m < mm && s_del[m] == 0;
        const unsigned ballot = __ballot_sync(kAll, keep);
        if (keep) s_pa[nk + __popc(ballot & lt_mask)] = m;
        nk += __popc(ballot);
    }
    __syncwarp();
    int off = 0;
    if (lane == 0) {        // the row allocation's round trip to L2 runs beside the ranking below
        off = atomicAdd(out_total, nk);
        out_offset[img] = off;
        out_count[img] = nk;
        redo[img] = 0;
    }
#pragma unroll 1
    for (int q = lane; q < nk; q += 32) {
        double ps = s_ps[s_pa[q]];
        if (ps != ps) ps = -1.0e300;        // documented deviation: NaN scores sort last
        int rank = 0;
#pragma unroll 1
        for (int q2 = 0; q2 < nk; ++q2) {
            double p2 = s_ps[s_pa[q2]];
            if (p2 != p2) p2 = -1.0e300;
            rank += (p2 > ps || (p2 == ps && q2 < q)) ? 1 : 0;
        }
        s_pb[q] = rank;
    }
    off = __shfl_sync(kAll, off, 0);
    __syncwarp();
    OG_K3_PROF(7);
    const float inv_c = __frcp_rn((float)C);
#pragma unroll 1
    for (int e = lane; e < nk * C; e += 32) {       // one lane per (person, joint): 24 bytes each
        const int q = small_div(e, inv_c), c = e - q * C;
        const int dst = off + s_pb[q];
        if (dst >= capacity_rows) continue;
        const int row = (int)s_order[s_pa[q]] * CS;
        const float4 v = xyvs[row + c];
        float2 *o = reinterpret_cast<float2 *>(out_poses + ((size_t)dst * C + c) * OG_POSE_COLS);
        o[0] = make_float2(unset_to_zero(v.x), unset_to_zero(v.y));
        o[1] = make_float2(unset_to_zero(v.z), unset_to_zero(v.w));
        o[2] = make_float2(unset_to_zero(score[row + c]), unset_to_zero((float)ids[row + c]));
        if (a.coco.frames != nullptr) {
            coco_joint(a.coco.frames + (size_t)(a.coco.image0 + img) * 4, unset_to_zero(v.x), unset_to_zero(v.y),
                       a.coco.keypoints + ((size_t)dst * C + c) * 3);
            if (c == 0) {       // score = sum(v) / len(v), float64, left to right (evaluate.py:250)
                double acc = 0.0;
#pragma unroll 1
                for (int cc = 0; cc < C; ++cc) acc += (double)unset_to_zero(xyvs[row + cc].z);
                a.coco.scores[dst] = acc / (double)C;
                a.coco.images[dst] = a.coco.image0 + img;
            }
        }
    }
#ifdef OG_K3_PROFILE
    OG_K3_PROF(8);
    if (threadIdx.x == 0) {
        for (int ph = 0; ph < 10; ++ph) atomicAdd(&og_k3_prof[ph], (unsigned long long)prof_acc[ph]);
        atomicAdd(&og_k3_prof[15], 1ull);
    }
#endif
}

GroupArgs to_args(const GroupLaunch &g) {
    GroupArgs a;
    a.C = g.c;
    a.L = g.l;
    a.K = g.k;
    a.sk = g.sk;
    a.person_thre = g.person_thre;
    a.sort_dim = g.sort_dim;
    a.warp_rows = g.warp_rows;
    a.slab = g.slab;
    a.slab_stride = g.slab_stride;
    a.coco = g.coco;
    a.lazy_flag = g.lazy_flag;
    return a;
}

}  // namespace

int read_k3_profile(unsigned long long *out16, bool reset) {
#ifdef OG_K3_PROFILE
    OG_CUDA_TRY(cudaMemcpyFromSymbol(out16, og_k3_prof, sizeof(unsigned long long) * 16));
    if (reset) {
        unsigned long long zeros[16] = {0};
        OG_CUDA_TRY(cudaMemcpyToSymbol(og_k3_prof, zeros, sizeof(zeros)));
    }
    return OG_OK;
#else
    (void)out16;
    (void)reset;
    set_error("library built without -DOG_K3_PROFILE");
    return OG_ERR_UNSUPPORTED;
#endif
}

size_t group_smem_bytes(const GroupLaunch &g) { return make_layout(g.l, g.k).total; }

size_t group_warp_smem_bytes(const GroupLaunch &g) {
    return g.warp_rows > 0 ? make_warp_layout(g.c, g.l, g.k, g.warp_rows).total : 0;
}

size_t group_prep_ints(const GroupLaunch &g) { return (size_t)g.n * g.l * (g.k + 1); }

size_t group_rec_vec4(const GroupLaunch &g) { return (size_t)g.n * g.l * g.k * 3; }

// The attributes belong to the kernels (per device), not to a handle: handles with different
// table sizes coexist, so they are only ever raised.
int prepare_group_kernel(size_t smem_bytes, size_t warp_smem_bytes) {
    static std::mutex mu;
    static size_t granted[64] = {0}, granted_warp[64] = {0};
    int dev = 0;
    OG_CUDA_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    const bool known = dev >= 0 && dev < 64;
    if (!known || smem_bytes > granted[dev]) {
        OG_CUDA_TRY(cudaFuncSetAttribute(group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem_bytes));
        if (known) granted[dev] = smem_bytes;
    }
    if (warp_smem_bytes > 48 * 1024 && (!known || warp_smem_bytes > granted_warp[dev])) {
        OG_CUDA_TRY(cudaFuncSetAttribute(group_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)warp_smem_bytes));
        if (known) granted_warp[dev] = warp_smem_bytes;
    }
    return OG_OK;
}

int launch_group(const GroupLaunch &g, const float *limbs, bool prepared, float *out_poses,
                 int capacity_rows, int32_t *out_offset, int32_t *out_count, int32_t *out_total,
                 cudaStream_t s, int64_t *launches) {
    if (g.n == 0) return OG_OK;
    if (!prepared) {
        prefer_chain_carveout<group_prepare_kernel>();
        group_prepare_kernel<<<dim3(g.l, g.n), kPrepThreads, 0, s>>>(limbs, g.l, g.k, g.dist_max,
                                                                     g.use_scale, g.prep, g.rec, g.cnt);
        OG_CUDA_TRY(cudaGetLastError());
        if (launches) *launches += 1;
    }
    if (g.warp_rows > 0) {
        prefer_chain_carveout<group_warp_kernel>();
        group_warp_kernel<<<g.n, 32, group_warp_smem_bytes(g), s>>>(
            to_args(g), g.rec, g.cnt, out_poses, capacity_rows, out_offset, out_count, out_total, g.redo);
        OG_CUDA_TRY(cudaGetLastError());
        if (launches) *launches += 1;
        // lazy: the caller looks at *lazy_flag once the launch has finished and calls
        // launch_group_redo for the (noise-like) batches that need it
        if (g.lazy_flag != nullptr) return OG_OK;
    }
    return launch_group_redo(g, limbs, out_poses, capacity_rows, out_offset, out_count, out_total, s, launches);
}

int launch_group_redo(const GroupLaunch &g, const float *limbs, float *out_poses, int capacity_rows,
                      int32_t *out_offset, int32_t *out_count, int32_t *out_total, cudaStream_t s,
                      int64_t *launches) {
    if (g.n == 0) return OG_OK;
    GroupLaunch cta = g;
    cta.lazy_flag = nullptr;
    prefer_chain_carveout<group_kernel>();
    group_kernel<<<g.n, kGroupThreads, group_smem_bytes(g), s>>>(
        to_args(cta), limbs, g.prep, out_poses, capacity_rows, out_offset, out_count, out_total,
        g.warp_rows > 0 ? g.redo : nullptr);
    OG_CUDA_TRY(cudaGetLastError());
    if (launches) *launches += 1;
    return OG_OK;
}

}  // namespace og
