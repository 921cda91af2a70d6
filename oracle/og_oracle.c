/*
 * TEST INFRASTRUCTURE — plain C (+ OpenMP) restatement of the reference's
 * post-network decoding path.  Only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may use it; the product library never links it.
 *
 * It follows the same reference lines as oracle/ref_oracle.py (which is pinned to the
 * reference's own outputs in tests/golden/) and is itself checked against those golden
 * fixtures by tests/test_c_oracle.py.  Unlike the numpy version it uses a real fmaf, so
 * it is bit-exact against ATen's CPU resize at every size, and it is fast enough to be
 * the CPU baseline and the full-size checker.
 *
 * Citations are relative to the reference repository (hellojialee/OffsetGuided):
 *   decoder/heatmap.py:15-49     oc_nms_topk
 *   decoder/collect.py:93-233    oc_limbs
 *   decoder/group.py:39-240      oc_group_image
 *   decoder/factory.py:98-146    oc_flip_fuse
 *   decoder/factory.py:74-78     oc_resize (ATen upsample_bicubic2d / upsample_bilinear2d,
 *                                align_corners=False, generic CPU kernel)
 *
 * Build: gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC (oracle/build_oracle.py).
 * -ffp-contract=off: fused multiply-adds happen only where fmaf() is written.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define LIMB_COLS 13
#define POSE_COLS 6

void oc_set_num_threads(int n) {
#ifdef _OPENMP
    if (n > 0) omp_set_num_threads(n);
#else
    (void)n;
#endif
}

int oc_num_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

/* ---------------------------------------------------------------- factory.py:98-146 */
void oc_flip_fuse(const float *hmp2n, const float *off2n, const int32_t *kp_flip,
                  const int32_t *limb_flip, const int32_t *limb_reserve, int n_reserve,
                  int n, int c, int l, int h, int w, float *out_h, float *out_o) {
    const long hw = (long)h * w;
    uint8_t reserved[256] = {0};
    for (int i = 0; i < n_reserve; ++i) reserved[limb_reserve[i]] = 1;
#pragma omp parallel for collapse(2) schedule(static)
    for (int img = 0; img < n; ++img)
        for (int ch = 0; ch < c; ++ch) {
            const float *a = hmp2n + ((long)img * c + ch) * hw;
            const float *b = hmp2n + ((long)(n + img) * c + kp_flip[ch]) * hw;
            float *o = out_h + ((long)img * c + ch) * hw;
            for (int y = 0; y < h; ++y)
                for (int x = 0; x < w; ++x)
                    o[y * w + x] = (a[y * w + x] + b[y * w + (w - 1 - x)]) / 2.0f;       /* :106 */
        }
#pragma omp parallel for collapse(2) schedule(static)
    for (int img = 0; img < n; ++img)
        for (int ch = 0; ch < 2 * l; ++ch) {
            const int limb = ch >> 1, comp = ch & 1;
            const float *a = off2n + ((long)img * 2 * l + ch) * hw;
            float *o = out_o + ((long)img * 2 * l + ch) * hw;
            if (reserved[limb]) {                                                        /* :134 */
                memcpy(o, a, sizeof(float) * hw);
                continue;
            }
            const float *b = off2n + ((long)(n + img) * 2 * l + 2 * limb_flip[limb] + comp) * hw;
            const float sign = comp == 0 ? -1.0f : 1.0f;                                  /* :132 */
            for (int y = 0; y < h; ++y)
                for (int x = 0; x < w; ++x)
                    o[y * w + x] = (a[y * w + x] + sign * b[y * w + (w - 1 - x)]) / 2.0f;  /* :133 */
        }
}

/* ---------------------------------------------------------------- factory.py:74-78 */
static void cubic_weights(float t, float w[4]) {
    const float A = -0.75f;
    const float x0 = t + 1.0f, x2 = 1.0f - t, x3 = 2.0f - t;
    w[0] = ((A * x0 - 5.0f * A) * x0 + 8.0f * A) * x0 - 4.0f * A;
    w[1] = ((A + 2.0f) * t - (A + 3.0f)) * t * t + 1.0f;
    w[2] = ((A + 2.0f) * x2 - (A + 3.0f)) * x2 * x2 + 1.0f;
    w[3] = ((A * x3 - 5.0f * A) * x3 + 8.0f * A) * x3 - 4.0f * A;
}

static int axis_taps(int dst, int n_in, float inv_scale, int cubic, int idx[4], float w[4]) {
    float real = inv_scale * ((float)dst + 0.5f) - 0.5f;
    if (!cubic && real < 0.0f) real = 0.0f;
    const float fl = floorf(real);
    const int base = (int)fl;
    float t = real - fl;
    if (t < 0.0f) t = 0.0f;
    if (t > 1.0f) t = 1.0f;
    if (cubic) {
        cubic_weights(t, w);
        for (int j = 0; j < 4; ++j) {
            int i = base + j - 1;
            idx[j] = i < 0 ? 0 : (i > n_in - 1 ? n_in - 1 : i);
        }
        return 4;
    }
    idx[0] = base < n_in - 1 ? base : n_in - 1;
    idx[1] = base + 1 < n_in - 1 ? base + 1 : n_in - 1;
    w[0] = 1.0f - t;
    w[1] = t;
    return 2;
}

/* accumulation order of ATen's generic interpolation loop as compiled with FMA
 * contraction (probed): round(t1*w1), fma(t0,w0,.), fma(t2,w2,.), fma(t3,w3,.) */
static inline float combine(const float *v, const float *w, int taps) {
    float acc = v[1] * w[1];
    acc = fmaf(v[0], w[0], acc);
    for (int j = 2; j < taps; ++j) acc = fmaf(v[j], w[j], acc);
    return acc;
}

void oc_resize(const float *in, float *out, int planes, int h, int w, int scale, int cubic) {
    const int oh = h * scale, ow = w * scale;
    const float inv = 1.0f / (float)scale;
    int *ix = (int *)malloc(sizeof(int) * 4 * ow);
    float *wx = (float *)malloc(sizeof(float) * 4 * ow);
    int taps = 2;
    for (int x = 0; x < ow; ++x) taps = axis_taps(x, w, inv, cubic, ix + 4 * x, wx + 4 * x);
#pragma omp parallel for collapse(2) schedule(static)
    for (int pl = 0; pl < planes; ++pl)
        for (int oy = 0; oy < oh; ++oy) {
            const float *p = in + (long)pl * h * w;
            float *o = out + ((long)pl * oh + oy) * ow;
            int iy[4];
            float wy[4];
            axis_taps(oy, h, inv, cubic, iy, wy);
            for (int ox = 0; ox < ow; ++ox) {
                float rows[4];
                for (int j = 0; j < taps; ++j) {
                    float v[4];
                    for (int i = 0; i < taps; ++i) v[i] = p[iy[j] * w + ix[4 * ox + i]];
                    rows[j] = combine(v, wx + 4 * ox, taps);
                }
                o[ox] = combine(rows, wy, taps);
            }
        }
    free(ix);
    free(wx);
}

/* ---------------------------------------------------------------- heatmap.py:15-49 */
/* Exact top-K of the NMS map (heat * (maxpool3x3_zero_pad == heat)), ordered
 * (value desc, flat index asc).  out_score / out_index are [planes][K]. */
void oc_nms_topk(const float *heat, int planes, int h, int w, int k, float *out_score,
                 int64_t *out_index) {
#pragma omp parallel for schedule(dynamic, 1)
    for (int pl = 0; pl < planes; ++pl) {
        const float *p = heat + (long)pl * h * w;
        float *bs = out_score + (long)pl * k;
        int64_t *bi = out_index + (long)pl * k;
        int cnt = 0;
        for (int y = 0; y < h; ++y)
            for (int x = 0; x < w; ++x) {
                const float v = p[y * w + x];
                float m = (y == 0 || x == 0 || y == h - 1 || x == w - 1) ? 0.0f : v;
                for (int dy = -1; dy <= 1; ++dy) {
                    const int yy = y + dy;
                    if (yy < 0 || yy >= h) continue;
                    for (int dx = -1; dx <= 1; ++dx) {
                        const int xx = x + dx;
                        if (xx < 0 || xx >= w) continue;
                        const float q = p[yy * w + xx];
                        if (q > m) m = q;
                    }
                }
                const float nv = v * ((m == v) ? 1.0f : 0.0f) + 0.0f;       /* heatmap.py:33-35 */
                /* insert into the sorted buffer; scanning in index order keeps ties index-asc */
                if (cnt == k && !(nv > bs[k - 1])) continue;
                int pos = cnt < k ? cnt : k - 1;
                while (pos > 0 && nv > bs[pos - 1]) {
                    bs[pos] = bs[pos - 1];
                    bi[pos] = bi[pos - 1];
                    --pos;
                }
                bs[pos] = nv;
                bi[pos] = (int64_t)y * w + x;
                if (cnt < k) ++cnt;
            }
    }
}

/* ---------------------------------------------------------------- collect.py:93-233 */
static inline float norm2(float dx, float dy) { return sqrtf(fmaf(dy, dy, dx * dx)); }

void oc_limbs(const float *det_score, const int64_t *det_index, const float *offs,
              const float *scales, int n, int c, int l, int k, int h, int w,
              const int32_t *from, const int32_t *to, float thre_hmp, float min_len,
              float resize_factor, float *out_limbs) {
    const long hw = (long)h * w;
#pragma omp parallel for collapse(2) schedule(static)
    for (int img = 0; img < n; ++img)
        for (int li = 0; li < l; ++li) {
            const int jf = from[li], jt = to[li];
            float tx[256], ty[256];
            const float *ss_t = det_score + ((long)img * c + jt) * k;
            const int64_t *ii_t = det_index + ((long)img * c + jt) * k;
            for (int m = 0; m < k; ++m) {                                   /* collect.py:247-254 */
                long xi = ii_t[m] % w, yi = ii_t[m] / w;
                if (ss_t[m] < thre_hmp) { xi -= 100000; yi -= 100000; }
                tx[m] = (float)xi;
                ty[m] = (float)yi;
            }
            const float *ss_f = det_score + ((long)img * c + jf) * k;
            const int64_t *ii_f = det_index + ((long)img * c + jf) * k;
            for (int q = 0; q < k; ++q) {
                long xi = ii_f[q] % w, yi = ii_f[q] / w;
                if (ss_f[q] < thre_hmp) { xi -= 100000; yi -= 100000; }
                const float x1 = (float)xi, y1 = (float)yi, s1 = ss_f[q];
                const float *o2 = offs + ((long)img * 2 * l + 2 * li) * hw + ii_f[q];   /* :143-147 */
                const float gx = x1 + o2[0] * resize_factor;                         /* :152 */
                const float gy = y1 + o2[hw] * resize_factor;
                float best = norm2(gx - tx[0], gy - ty[0]);
                int bm = 0;
                for (int m = 1; m < k; ++m) {                                         /* :171-177 */
                    const float d = norm2(gx - tx[m], gy - ty[m]);
                    if (d < best) { best = d; bm = m; }
                }
                float len = norm2(x1 - tx[bm], y1 - ty[bm]);                        /* :204 */
                if (len < min_len) len = min_len;
                float sc1 = 4.0f, sc2 = 4.0f;                                        /* :117-122 */
                if (scales) {
                    sc1 = scales[((long)img * c + jf) * hw + ii_f[q]];
                    sc2 = scales[((long)img * c + jt) * hw + ii_t[bm]];
                }
                float *o = out_limbs + (((long)img * l + li) * k + q) * LIMB_COLS;
                o[0] = x1; o[1] = y1; o[2] = s1;
                o[3] = tx[bm]; o[4] = ty[bm]; o[5] = ss_t[bm];
                o[6] = (float)(ii_f[q] + (int64_t)jf * hw);                          /* :198-199 */
                o[7] = (float)(ii_t[bm] + (int64_t)jt * hw);
                o[8] = best; o[9] = len;
                o[10] = s1 * ss_t[bm] * expf(-best / len);                            /* :208 */
                o[11] = sc1; o[12] = sc2;
            }
        }
}

/* ---------------------------------------------------------------- group.py:39-240 */
static float numpy_sum_f32(const float *a, int n) {       /* numpy pairwise sum, n <= 128 */
    if (n < 8) {
        float s = 0.0f;
        for (int i = 0; i < n; ++i) s += a[i];
        return s;
    }
    float r[8];
    for (int j = 0; j < 8; ++j) r[j] = a[j];
    int i = 8;
    for (; i < n - (n % 8); i += 8)
        for (int j = 0; j < 8; ++j) r[j] += a[i + j];
    float s = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) s += a[i];
    return s;
}

#define S(m, j, f) subset[((long)(m) * c + (j)) * POSE_COLS + (f)]

/* limbs [L][K][13] -> out [<= L*K][C][6]; returns the number of persons */
int oc_group_image(const float *limbs, int c, int l, int k, const int32_t *from,
                   const int32_t *to, float dist_max, int use_scale, double person_thre,
                   int sort_dim, float *out) {
    const int pmax = l * k;
    float *subset = (float *)malloc(sizeof(float) * (size_t)pmax * c * POSE_COLS);
    float *rowtmp = (float *)malloc(sizeof(float) * (size_t)pmax * c * POSE_COLS);
    int *msum = (int *)malloc(sizeof(int) * (size_t)pmax * k);
    uint8_t *repl = (uint8_t *)malloc((size_t)pmax * k);
    int *pm = (int *)malloc(sizeof(int) * (size_t)pmax * (k > pmax ? k : pmax));
    int *pk = (int *)malloc(sizeof(int) * (size_t)pmax * (k > pmax ? k : pmax));
    float *rhs = (float *)malloc(sizeof(float) * (size_t)pmax * k);
    int *id_f = (int *)malloc(sizeof(int) * pmax), *id_t = (int *)malloc(sizeof(int) * pmax);
    float *sc_f = (float *)malloc(sizeof(float) * pmax), *sc_t = (float *)malloc(sizeof(float) * pmax);
    uint8_t *gone = (uint8_t *)malloc(pmax);
    int rows[256], kept[256];
    int mm = 0;

    for (int li = 0; li < l; ++li) {
        const int jf = from[li], jt = to[li];
        const float *conns = limbs + (long)li * k * LIMB_COLS;
        int nv = 0;
        for (int q = 0; q < k; ++q) {                                           /* :64-76 */
            const float *r = conns + q * LIMB_COLS;
            float lim = dist_max;
            if (use_scale) lim = (r[12] != r[12]) ? r[12] : (dist_max > r[12] ? dist_max : r[12]);
            if (r[8] < lim && r[0] > 0 && r[4] > 0 && r[3] > 0 && r[1] > 0) rows[nv++] = q;
        }
        /* stable sort, limb score desc (:232); NaN scores (0 / 0 at min_len = 0) after every
         * number, in row order: the stable form of np.argsort(-s) */
        for (int i = 1; i < nv; ++i) {
            const int q = rows[i];
            const float s = conns[q * LIMB_COLS + 10];
            int j = i - 1;
            while (j >= 0 && s == s) {
                const float t = conns[rows[j] * LIMB_COLS + 10];
                if (!(t != t || t < s)) break;
                rows[j + 1] = rows[j];
                --j;
            }
            rows[j + 1] = q;
        }
        int kk = 0;
        for (int i = 0; i < nv; ++i) {                                          /* :233-239 */
            const int t = (int)conns[rows[i] * LIMB_COLS + 7];
            int dup = 0;
            for (int j = 0; j < kk && !dup; ++j) dup = ((int)conns[kept[j] * LIMB_COLS + 7] == t);
            if (!dup) kept[kk++] = rows[i];
        }
        if (kk == 0) continue;                                                  /* :84-85 */

        for (int m = 0; m < mm; ++m) {                                          /* :87-88 */
            id_f[m] = (int)S(m, jf, 5); id_t[m] = (int)S(m, jt, 5);
            sc_f[m] = S(m, jf, 4);      sc_t[m] = S(m, jt, 4);
        }
        for (int m = 0; m < mm; ++m)
            for (int q = 0; q < kk; ++q) {
                const float *r = conns + kept[q] * LIMB_COLS;
                msum[m * kk + q] = (id_f[m] == (int)r[6]) + (id_t[m] == (int)r[7]);   /* :103-104 */
                repl[m * kk + q] = (r[10] > sc_t[m]) || (r[10] > sc_f[m]);            /* :108-109 */
            }
        for (int which = 2; which >= 1; --which) {           /* :114-119 then :124-135 */
            int np_ = 0;
            for (int m = 0; m < mm; ++m)
                for (int q = 0; q < kk; ++q)
                    if (msum[m * kk + q] == which && repl[m * kk + q]) { pm[np_] = m; pk[np_] = q; ++np_; }
            if (!np_) continue;
            if (which == 1) {
                for (int i = 0; i < np_; ++i) S(pm[i], jf, 5) = conns[kept[pk[i]] * LIMB_COLS + 6];
                for (int i = 0; i < np_; ++i) S(pm[i], jt, 5) = conns[kept[pk[i]] * LIMB_COLS + 7];
                for (int i = 0; i < np_; ++i) {
                    const float *r = conns + kept[pk[i]] * LIMB_COLS;
                    S(pm[i], jf, 0) = r[0]; S(pm[i], jf, 1) = r[1]; S(pm[i], jf, 2) = r[2]; S(pm[i], jf, 3) = r[11];
                }
                for (int i = 0; i < np_; ++i) {
                    const float *r = conns + kept[pk[i]] * LIMB_COLS;
                    S(pm[i], jt, 0) = r[3]; S(pm[i], jt, 1) = r[4]; S(pm[i], jt, 2) = r[5]; S(pm[i], jt, 3) = r[12];
                }
            }
            const int joints[2] = {jf, jt};
            for (int e = 0; e < 2; ++e) {        /* right-hand side first, then scatter in order */
                for (int i = 0; i < np_; ++i) {
                    const float s = conns[kept[pk[i]] * LIMB_COLS + 10];
                    const float cur = S(pm[i], joints[e], 4);
                    rhs[i] = s > cur ? s : cur;
                }
                for (int i = 0; i < np_; ++i) S(pm[i], joints[e], 4) = rhs[i];
            }
            for (int i = 0; i < mm * kk; ++i)
                if (msum[i] == which) msum[i] = -1;
        }
        int mm_after = mm;
        if (mm >= 2) {                                                           /* :140-155 */
            int np_ = 0;
            for (int a = 0; a < mm; ++a)
                for (int b = a + 1; b < mm; ++b) {
                    int shared = 0;
                    for (int j = 0; j < c; ++j) {
                        const int ia = (int)S(a, j, 5);
                        shared += (ia != -1 && ia == (int)S(b, j, 5));
                    }
                    if (shared == 2) { pm[np_] = a; pk[np_] = b; ++np_; }
                }
            if (np_) {
                /* right-hand sides read the pre-merge rows; for duplicate targets the
                 * last pair (largest partner) wins */
                const int rs = c * POSE_COLS;
                memcpy(rowtmp, subset, sizeof(float) * (size_t)mm * rs);
                for (int i = 0; i < np_; ++i)
                    for (int e = 0; e < rs; ++e) {
                        const float x = rowtmp[(long)pm[i] * rs + e], y = rowtmp[(long)pk[i] * rs + e];
                        subset[(long)pm[i] * rs + e] = x > y ? x : y;
                    }
                memset(gone, 0, mm);
                for (int i = 0; i < np_; ++i) gone[pk[i]] = 1;
                int w_ = 0;
                for (int m = 0; m < mm; ++m)
                    if (!gone[m]) {
                        if (w_ != m) memmove(subset + (long)w_ * rs, subset + (long)m * rs, sizeof(float) * rs);
                        ++w_;
                    }
                mm_after = w_;
            }
        }
        for (int q = 0; q < kk; ++q) {                                           /* :166-177 */
            int col = 0;
            for (int m = 0; m < mm; ++m) col += msum[m * kk + q];
            if (col != 0) continue;
            const float *r = conns + kept[q] * LIMB_COLS;
            for (int e = 0; e < c * POSE_COLS; ++e) subset[(long)mm_after * c * POSE_COLS + e] = -1.0f;
            S(mm_after, jf, 5) = r[6]; S(mm_after, jt, 5) = r[7];
            S(mm_after, jf, 0) = r[0]; S(mm_after, jf, 1) = r[1]; S(mm_after, jf, 2) = r[2]; S(mm_after, jf, 3) = r[11];
            S(mm_after, jt, 0) = r[3]; S(mm_after, jt, 1) = r[4]; S(mm_after, jt, 2) = r[5]; S(mm_after, jt, 3) = r[12];
            S(mm_after, jf, 4) = r[10]; S(mm_after, jt, 4) = r[10];
            ++mm_after;
        }
        mm = mm_after;
    }

    /* _delete_sort (:188-219) */
    double *ps = (double *)malloc(sizeof(double) * (mm > 0 ? mm : 1));
    int *order = (int *)malloc(sizeof(int) * (mm > 0 ? mm : 1));
    int nk = 0;
    for (int m = 0; m < mm; ++m) {
        float vals[256];
        int nvv = 0;
        for (int j = 0; j < c; ++j)
            if (S(m, j, sort_dim) > 0) vals[nvv++] = S(m, j, sort_dim);
        const double s = (double)numpy_sum_f32(vals, nvv) / (double)nvv;
        if (s < person_thre) continue;
        ps[nk] = s;
        order[nk] = m;
        ++nk;
    }
    for (int i = 1; i < nk; ++i) {          /* stable descending */
        const int m = order[i];
        const double s = ps[i];
        int j = i - 1;
        while (j >= 0 && ps[j] < s) { ps[j + 1] = ps[j]; order[j + 1] = order[j]; --j; }
        ps[j + 1] = s;
        order[j + 1] = m;
    }
    for (int i = 0; i < nk; ++i)
        for (int e = 0; e < c * POSE_COLS; ++e) {
            const float v = subset[(long)order[i] * c * POSE_COLS + e];
            out[(long)i * c * POSE_COLS + e] = (v == -1.0f) ? 0.0f : v;
        }
    free(ps); free(order); free(subset); free(rowtmp); free(msum); free(repl); free(pm); free(pk);
    free(rhs); free(id_f); free(id_t); free(sc_f); free(sc_t); free(gone);
    return nk;
}

/* all images of a batch in parallel; out [n][L*K][C][6], counts [n] */
void oc_group_batch(const float *limbs, int n, int c, int l, int k, const int32_t *from,
                    const int32_t *to, float dist_max, int use_scale, double person_thre,
                    int sort_dim, float *out, int32_t *counts) {
#pragma omp parallel for schedule(dynamic, 1)
    for (int img = 0; img < n; ++img)
        counts[img] = oc_group_image(limbs + (long)img * l * k * LIMB_COLS, c, l, k, from, to,
                                     dist_max, use_scale, person_thre, sort_dim,
                                     out + (long)img * l * k * c * POSE_COLS);
}
